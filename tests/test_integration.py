"""The compiled drop-in: oracle/_ref/snap-aligner-gpu = the UNMODIFIED reference (SNAPLib objects) linked with
integration/GpuAlignerExtension.cpp and libsnapgpu.so.  `snap-aligner-gpu single|paired <index> reads.fq -o out.sam` must write the
records stock `snap-aligner` writes for the same command line -- the reference's own option parser, FASTQ reader, filter and SAM
writer run on both sides; only the aligner behind AlignerExtension::runIterationThread differs."""
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GPU_BIN = os.path.join(ROOT, "oracle", "_ref", "snap-aligner-gpu")


def test_binding_is_built_and_links_the_product_library():
    """CPU-side: the binary exists (built by __graft_entry__.build() where the reference sources are present) and its only non-system
    dependency is libsnapgpu.so; no compute here."""
    if not os.path.exists(GPU_BIN):
        pytest.skip("oracle/_ref/snap-aligner-gpu not built (needs the reference sources once: make -C oracle ref)")
    out = subprocess.run(["ldd", GPU_BIN], capture_output=True, text=True).stdout
    assert "libsnapgpu.so" in out and "not found" not in out, out
    assert "libsnapref" not in out            # the oracle shim is not part of the drop-in
    src = open(os.path.join(ROOT, "integration", "GpuAlignerExtension.cpp")).read()
    for sym in ("snapgpu_align_single", "snapgpu_align_paired", "snapgpu_index_open", "snapgpu_index_broadcast", "snapgpu_counters_allreduce", "snapgpu_aligner_create",
                "snapgpu_paired_aligner_create"):
        assert sym in src


def _records(path):
    return sorted(l for l in open(path, "rb").read().split(b"\n") if l and not l.startswith(b"@"))


def _run(binary, argv, env=None):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([binary] + argv, capture_output=True, text=True, env=e, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


def _stats_line(stdout, n=5):
    lines = [l for l in stdout.split("\n") if l.strip()]
    k = max(i for i, l in enumerate(lines) if "Reads/s" in l)
    import re
    toks = re.sub(r"\([^)]*\)", " ", lines[k + 1]).split()
    return [t for t in toks if t.replace(",", "").isdigit()][:n]       # total, single, multi, unaligned, too short[, extra alignments] (rates / times differ)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 4])
def test_snap_aligner_gpu_single_writes_the_stock_records(tmp_path, small_cfg, reflib, threads):
    if not os.path.exists(GPU_BIN):
        pytest.fail("oracle/_ref/snap-aligner-gpu is missing")
    from snap_b200 import synth
    reads = small_cfg.reads["noisy150"]           # N runs, short reads, noise, indels
    fq = str(tmp_path / "r.fq")
    reads.write_fastq(fq)
    stock, gpu = str(tmp_path / "stock.sam"), str(tmp_path / "gpu.sam")
    so = _run(reflib.SNAP_ALIGNER, ["single", small_cfg.idx, fq, "-o", stock, "-t", "1", "-d", "14"])
    go = _run(GPU_BIN, ["single", small_cfg.idx, fq, "-o", gpu, "-t", str(threads), "-d", "14"], env={"SNAPGPU_EXT_BATCH_READS": "512"})
    a, b = _records(stock), _records(gpu)
    assert len(a) == reads.n and len(b) == reads.n
    bad = [i for i in range(len(a)) if a[i] != b[i]]
    assert not bad, (len(bad), a[bad[0]], b[bad[0]])
    assert _stats_line(so) == _stats_line(go)          # printStats totals (AlignerContext.cpp:491-540)
    assert "CUDA device" in go


@pytest.mark.gpu
def test_snap_aligner_gpu_single_other_options(tmp_path, small_cfg, reflib):
    """-d 20 -G- (no affine gap), -= (X/= CIGARs) and a filter: options travel through the reference's parser into snapgpu_params."""
    reads = small_cfg.reads["indel100"]
    fq = str(tmp_path / "r.fq")
    reads.write_fastq(fq)
    for extra in (["-d", "20", "-G-"], ["-d", "8", "-=", "-F", "a"], ["-d", "14", "-h", "20", "-D", "3"]):
        stock, gpu = str(tmp_path / "stock.sam"), str(tmp_path / "gpu.sam")
        _run(reflib.SNAP_ALIGNER, ["single", small_cfg.idx, fq, "-o", stock, "-t", "1"] + extra)
        _run(GPU_BIN, ["single", small_cfg.idx, fq, "-o", gpu, "-t", "2"] + extra)
        a, b = _records(stock), _records(gpu)
        assert a == b, (extra, len(a), len(b))


@pytest.mark.gpu
def test_snap_aligner_gpu_single_secondary_alignments(tmp_path, small_cfg, reflib):
    """`-om` (with -omax / -mpc): the records of the primary AND the secondary alignments (flag 0x100) are the ones stock snap-aligner writes,
    and so are the totals it prints (extra alignments included)."""
    reads = small_cfg.reads["std150"]
    fq = str(tmp_path / "r.fq")
    reads.write_fastq(fq)
    for extra in (["-d", "14", "-om", "1"], ["-d", "14", "-D", "3", "-om", "3", "-omax", "4"], ["-d", "14", "-D", "2", "-om", "2", "-mpc", "1", "-G-"]):
        stock, gpu = str(tmp_path / "stock.sam"), str(tmp_path / "gpu.sam")
        so = _run(reflib.SNAP_ALIGNER, ["single", small_cfg.idx, fq, "-o", stock, "-t", "1"] + extra)
        go = _run(GPU_BIN, ["single", small_cfg.idx, fq, "-o", gpu, "-t", "2"] + extra, env={"SNAPGPU_EXT_BATCH_READS": "512"})
        a, b = _records(stock), _records(gpu)
        assert len(a) > reads.n                    # there are secondary records
        assert a == b, (extra, len(a), len(b))
        assert _stats_line(so, 6) == _stats_line(go, 6) and int(_stats_line(so, 6)[5].replace(",", "")) == len(a) - reads.n


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 3])
def test_snap_aligner_gpu_paired_writes_the_stock_records(tmp_path, small_cfg, reflib, threads):
    if not os.path.exists(GPU_BIN):
        pytest.fail("oracle/_ref/snap-aligner-gpu is missing")
    pairs = small_cfg.pairs["std150"]             # chimeric mates, N runs, short ends
    f1, f2 = str(tmp_path / "r1.fq"), str(tmp_path / "r2.fq")
    with open(f1, "wb") as a, open(f2, "wb") as b:
        for i in range(pairs.n // 2):
            for w, f in ((0, a), (1, b)):
                bs, q = pairs.read(2 * i + w)
                f.write(b"@p%d/%d\n%s\n+\n%s\n" % (i, w + 1, bs, q))
    stock, gpu = str(tmp_path / "stock.sam"), str(tmp_path / "gpu.sam")
    so = _run(reflib.SNAP_ALIGNER, ["paired", small_cfg.idx, f1, f2, "-o", stock, "-t", "1"])
    go = _run(GPU_BIN, ["paired", small_cfg.idx, f1, f2, "-o", gpu, "-t", str(threads)], env={"SNAPGPU_EXT_BATCH_READS": "256"})
    x, y = _records(stock), _records(gpu)
    assert len(x) == pairs.n and len(y) == pairs.n
    bad = [i for i in range(len(x)) if x[i] != y[i]]
    assert not bad, (len(bad), x[bad[0]], y[bad[0]])
    assert _stats_line(so) == _stats_line(go)
