"""-m gpu: nvCOMP's OWN benchmarks and examples, compiled unchanged against include/ + libnvcomp.so, as the
acceptance harness: every one of them self-verifies (status, sizes, bytes) and prints the reference's report
(benchmarks/benchmark_template_chunked.cuh:553-617).

Their reports on a B200 are stored in tests/golden/reference_harness.json (tests/golden/make_reference_reports.py).
Every test replays its program's workload -- same bytes, same chunking, same format options -- through the same C
ABI and checks the result against that stored report, so the suite needs no nvCOMP sources.  Where
oracle/build_reference_harness.sh has built the programs into oracle/_ref/, the test also runs the program itself
and checks its fresh report against the stored one."""
import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
BIN = os.path.join(ROOT, "oracle", "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_harness.json")
CHUNK = 65536

CHUNKED = [("lz4", "f32", []), ("lz4", "i32", ["-t", "int"]), ("snappy", "f32", []),
           ("cascaded", "i64", ["-t", "longlong", "-r", "1", "-d", "1", "-b", "1"]), ("cascaded", "i32", ["-t", "int"]),
           ("bitcomp", "i64", ["-t", "ulonglong"]), ("bitcomp", "i32", ["-t", "uint", "-a", "1"]), ("ans", "bytes", [])]
HLIF = [("lz4", "f32", []), ("snappy", "i32", []), ("ans", "bytes", []), ("bitcomp", "i32", ["-t", "int"]),
        ("cascaded", "i32", ["-t", "int"])]
INTEROP_KEYS = ["f32", "i32", "bytes"]


def _runs():
    """golden key -> the program and its arguments; "{name}" stands for the data file write_data_files() made."""
    runs = {f"chunked:{f}:{k}:{' '.join(x)}": [f"benchmark_{f}_chunked", "-f", "{%s}" % k, *x] for f, k, x in CHUNKED}
    runs["snappy_synth:500"] = ["benchmark_snappy_synth", "-b", "500", "-w", "2", "-i", "3"]
    runs["snappy_synth:200"] = ["benchmark_snappy_synth", "-b", "200", "-w", "1", "-i", "2"]
    runs["lz4_synth"] = ["benchmark_lz4_synth"]
    for k in INTEROP_KEYS:
        runs[f"lz4_cpu_compression:{k}"] = ["lz4_cpu_compression", "-f", "{%s}" % k]
        runs[f"lz4_cpu_decompression:{k}"] = ["lz4_cpu_decompression", "-f", "{%s}" % k]
    runs["low_level_quickstart"] = ["low_level_quickstart_example"]
    runs["high_level_quickstart"] = ["high_level_quickstart_example"]
    runs.update({f"hlif:{f}:{k}:{' '.join(x)}": ["benchmark_hlif", f, "-f", "{%s}" % k, *x] for f, k, x in HLIF})
    runs["zstd_chunked:bytes"] = ["benchmark_zstd_chunked", "-f", "{bytes}"]
    return runs


RUNS = _runs()


def write_data_files(d) -> dict:
    from nvcomp_b200 import datagen
    files = {}
    for name, arr in (("i32", datagen.runlength_i32(64)), ("f32", datagen.tabular_f32(64)),
                      ("i64", datagen.sorted_i64(64)), ("bytes", datagen.lowentropy_bytes(64))):
        p = os.path.join(str(d), f"{name}.bin")
        arr.reshape(-1)[: 64 * 65536 - 1234 if name == "bytes" else None].tofile(p)
        files[name] = p
    return files


def parse_report(rc: int, out: str) -> dict:
    """The deterministic part of a report: exit status, byte counts, and the validation lines."""
    return {"ok": rc == 0,
            "uncompressed": [int(x) for x in re.findall(r"uncompressed \(B\): (\d+)", out)],
            "comp_size": [int(x) for x in re.findall(r"comp_size: (\d+)", out)],
            "validated": [ln.strip() for ln in out.splitlines() if "validated" in ln],
            "throughput_lines": out.count("decompression throughput (GB/s)")}


def run_program(key, files, timeout=900):
    prog, *args = RUNS[key]
    r = subprocess.run([os.path.join(BIN, prog), *[a.format(**files) for a in args]], capture_output=True, text=True,
                       timeout=timeout)
    return r.returncode, r.stdout, r.stderr


@pytest.fixture(scope="module")
def golden():
    return json.load(open(GOLDEN))


@pytest.fixture(scope="module")
def data_files(tmp_path_factory):
    return write_data_files(tmp_path_factory.mktemp("refdata"))


def _reference(key, golden, files, timeout=900) -> dict:
    """The stored report of run `key`; when its program was built, run it and require the same report."""
    want = golden[key]
    if os.path.exists(os.path.join(BIN, RUNS[key][0])):
        rc, out, err = run_program(key, files, timeout)
        assert parse_report(rc, out) == want, (key, out[-2000:], err[-2000:])
    return want


def _chunks(path, chunk=CHUNK):
    raw = open(path, "rb").read()
    return [raw[i:i + chunk] for i in range(0, len(raw), chunk)]


def _opts(fmt, extra):
    """The format options the nvCOMP benchmark programs build from their command line (their defaults first)."""
    from nvcomp_b200._lib import OPTS, Type
    types = {"char": Type.CHAR, "uchar": Type.UCHAR, "short": Type.SHORT, "ushort": Type.USHORT, "int": Type.INT,
             "uint": Type.UINT, "longlong": Type.LONGLONG, "ulonglong": Type.ULONGLONG}
    kw = dict(zip(extra[::2], extra[1::2]))
    t = types[kw["-t"]] if "-t" in kw else None
    if fmt == "lz4":
        return OPTS["LZ4"](Type.CHAR if t is None else t)
    if fmt == "cascaded":
        return OPTS["Cascaded"](4096, Type.UINT if t is None else t, int(kw.get("-r", 2)), int(kw.get("-d", 1)),
                                int(kw.get("-b", 1)))
    if fmt == "bitcomp":
        return OPTS["Bitcomp"](int(kw.get("-a", 0)), Type.UCHAR if t is None else t)
    return None


def _codec(fmt, extra=()):
    from nvcomp_b200.batched import Codec
    name = {"lz4": "LZ4", "snappy": "Snappy", "cascaded": "Cascaded", "bitcomp": "Bitcomp", "ans": "ANS"}[fmt]
    return Codec(name, opts=_opts(fmt, list(extra)))


def _roundtrip(codec, chunks):
    """GPU compress + GPU decompress of the chunks, bit-exact; returns the compressed streams."""
    from gpu_util import gpu_compress, gpu_decompress
    comps, _ = gpu_compress(codec, chunks)
    outs, actual, status, _ = gpu_decompress(codec, comps, [len(c) for c in chunks])
    assert (status == 0).all() and list(actual) == [len(c) for c in chunks] and outs == chunks
    return comps


@pytest.mark.parametrize("fmt,key,extra", CHUNKED)
def test_chunked_benchmarks(fmt, key, extra, data_files, golden):
    """benchmark_<fmt>_chunked -f file: compress -> decompress -> byte compare inside the reference harness."""
    want = _reference(f"chunked:{fmt}:{key}:{' '.join(extra)}", golden, data_files)
    assert want["ok"] and want["throughput_lines"] == 1
    chunks = _chunks(data_files[key])
    comps = _roundtrip(_codec(fmt, extra), chunks)
    assert [sum(map(len, chunks))] == want["uncompressed"]
    assert [sum(map(len, comps))] == want["comp_size"]


def test_snappy_synth(data_files, golden):
    """benchmark_snappy_synth -b 500: 500 chunks of the reference's gen_data(3) stream, Snappy round trip."""
    from nvcomp_b200 import datagen
    batch = 500
    want = _reference(f"snappy_synth:{batch}", golden, data_files)
    assert want["ok"] and want["throughput_lines"] == 1
    chunks = [r.tobytes() for r in datagen.snappy_synth(batch, 3)]
    comps = _roundtrip(_codec("snappy"), chunks)
    assert [batch * CHUNK] == want["uncompressed"] and [sum(map(len, comps))] == want["comp_size"]


def test_lz4_synth_hlif(data_files, golden):
    """benchmark_lz4_synth: LZ4Manager round trips of all-zero and all-random buffers, 64 KB ... 512 MB
    (reference benchmarks/benchmark_lz4_synth.cpp:64-72; BASELINE configs[0] names this path).  The replay sends the
    same buffer sizes through the batched LZ4 calls the manager is built on."""
    import torch
    from nvcomp_b200.batched import Batch, empty_batch
    want = _reference("lz4_synth", golden, data_files)
    sizes = [CHUNK << b for b in range(14)]
    assert want["ok"] and want["throughput_lines"] == 28 and want["uncompressed"] == sizes * 2
    codec = _codec("lz4")
    gen = torch.Generator(device="cuda").manual_seed(0)
    for random in (False, True):
        for size in sizes:
            n = size // CHUNK
            slab = (torch.randint(0, 256, (size,), dtype=torch.uint8, device="cuda", generator=gen) if random
                    else torch.zeros(size, dtype=torch.uint8, device="cuda"))
            offs = np.arange(n, dtype=np.int64) * CHUNK
            inp = Batch(slab, torch.from_numpy(offs + slab.data_ptr()).cuda(),
                        torch.full((n,), CHUNK, dtype=torch.int64, device="cuda"), offs)
            comp = codec.compress(inp, max_chunk=CHUNK)
            out = empty_batch(n, CHUNK, fill=0xA5)
            actual, status = codec.decompress(comp, out, max_chunk=CHUNK)
            torch.cuda.synchronize()
            assert bool((status == 0).all()) and bool((actual == CHUNK).all()), (random, size)
            assert torch.equal(out.slab[: size].view(n, CHUNK), slab.view(n, CHUNK)), (random, size)


@pytest.mark.parametrize("key", INTEROP_KEYS)
def test_lz4_cpu_interop_examples(key, data_files, golden, liblz4):
    """The reference's known-answer tests of the LZ4 wire format, compiled unchanged (tests/shim/lz4.h only declares
    liblz4's prototypes): liblz4-HC(12) streams decode on the GPU (examples/lz4_cpu_compression.cu:61-66,121-140) and
    GPU streams decode with LZ4_decompress_safe (examples/lz4_cpu_decompression.cu:143-157)."""
    from gpu_util import gpu_compress, gpu_decompress
    want = _reference(f"lz4_cpu_compression:{key}", golden, data_files)
    assert want["ok"] and want["validated"] == ["decompression validated :)"]
    chunks = _chunks(data_files[key])
    codec = _codec("lz4")
    hc = [liblz4.compress(c, 12) for c in chunks]
    outs, _, status, _ = gpu_decompress(codec, hc, [len(c) for c in chunks])
    assert (status == 0).all() and outs == chunks
    assert [sum(map(len, chunks))] == want["uncompressed"] and [sum(map(len, hc))] == want["comp_size"]

    want = _reference(f"lz4_cpu_decompression:{key}", golden, data_files)
    assert want["ok"] and want["validated"] == ["CPU decompression validated :)"]
    comps, _ = gpu_compress(codec, chunks)
    assert [liblz4.decompress(c, CHUNK) for c in comps] == chunks
    assert [sum(map(len, chunks))] == want["uncompressed"] and [sum(map(len, comps))] == want["comp_size"]


def test_quickstarts(data_files, golden):
    """examples/{low,high}_level_quickstart_example: LZ4 round trip of 1,000,000 random bytes in 64 KB chunks."""
    for key in ("low_level_quickstart", "high_level_quickstart"):
        assert _reference(key, golden, data_files)["ok"], key
    raw = np.random.default_rng(42).integers(0, 256, 1000000, dtype=np.uint8).tobytes()
    _roundtrip(_codec("lz4"), [raw[i:i + CHUNK] for i in range(0, len(raw), CHUNK)])


@pytest.mark.parametrize("fmt,key,extra", HLIF)
def test_hlif_benchmark(fmt, key, extra, data_files, golden):
    """benchmark_hlif <fmt> -f file: the format's manager over the whole file.  The replay sends the file through the
    batched calls of the same format and data type."""
    want = _reference(f"hlif:{fmt}:{key}:{' '.join(extra)}", golden, data_files)
    assert want["ok"] and want["throughput_lines"] == 1
    chunks = _chunks(data_files[key])
    _roundtrip(_codec(fmt, extra), chunks)
    assert [sum(map(len, chunks))] == want["uncompressed"]


def test_unsupported_formats_report_not_supported(data_files, golden):
    """benchmark_zstd_chunked: an out-of-scope format -- the harness' status assert on its first call
    (BatchedCompressGetTempSize) fires, nothing crashes."""
    from nvcomp_b200 import load

    class ZstdOpts(C.Structure):
        _fields_ = [("algo", C.c_int)]
    assert not _reference("zstd_chunked:bytes", golden, data_files, timeout=120)["ok"]
    out = C.c_size_t(0)
    fn = load().nvcompBatchedZstdCompressGetTempSize
    fn.argtypes, fn.restype = [C.c_size_t, C.c_size_t, ZstdOpts, C.POINTER(C.c_size_t)], C.c_int
    assert fn(len(_chunks(data_files["bytes"])), CHUNK, ZstdOpts(0), C.byref(out)) == 11     # nvcompErrorNotSupported


def test_cmake_built_reference_binary_runs(data_files, golden):
    """A binary produced by nvCOMP's OWN CMake build against cmake/nvcomp-config.cmake (INTEGRATION.md; build/ref_cmake,
    PTX-JIT from compute_90 on B200), when present; the replay is benchmark_snappy_synth -b 200."""
    from nvcomp_b200 import datagen
    exe = os.path.join(ROOT, "build", "ref_cmake", "bin", "low_level_quickstart_example")
    if os.path.exists(exe):
        r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
        exe = os.path.join(ROOT, "build", "ref_cmake", "bin", "benchmark_snappy_synth")
        r = subprocess.run([exe, "-b", "200", "-w", "1", "-i", "2"], capture_output=True, text=True, timeout=600)
        assert parse_report(r.returncode, r.stdout) == golden["snappy_synth:200"], (r.stdout[-2000:], r.stderr[-2000:])
    want = _reference("snappy_synth:200", golden, data_files)
    comps = _roundtrip(_codec("snappy"), [r.tobytes() for r in datagen.snappy_synth(200, 3)])
    assert want["ok"] and [sum(map(len, comps))] == want["comp_size"]
