"""JNI glue (jni/tsgpu_jni.c): compiled as it stands against a test-only stand-in for <jni.h> and driven through a fake
JNIEnv by tests/cpp/test_jni_shim.c (copy-in/copy-out array semantics, exception mapping, round trip checked by the
oracle); plus a check that every `native` method TsGpu.java declares has its Java_* export with the right arity."""
import json
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "io/aiven/kafka/tieredstorage/transform/gpu"


def test_jni_glue_through_a_fake_jnienv():
    subprocess.check_call(["make", "-s", "-C", ROOT, "tests/cpp/test_jni_shim_simt"], stderr=subprocess.DEVNULL)
    out = subprocess.run([os.path.join(ROOT, "tests/cpp/test_jni_shim_simt")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().splitlines()[-1].startswith("OK:"), out.stdout + out.stderr


def test_java_native_declarations_match_the_exports():
    java = open(os.path.join(ROOT, "jni", PKG, "TsGpu.java")).read()
    c = open(os.path.join(ROOT, "jni", "tsgpu_jni.c")).read()
    natives = re.findall(r"public static native\s+\S+\s+(\w+)\(([^)]*)\)", java, flags=re.S)
    assert len(natives) == 7
    for name, params in natives:
        m = re.search(r"Java_" + PKG.replace("/", "_") + "_TsGpu_" + name + r"\(([^)]*)\)", c, flags=re.S)
        assert m, name
        n_java = len([p for p in params.split(",") if p.strip()])
        n_c = len([p for p in m.group(1).split(",") if p.strip()])
        assert n_c == n_java + 2, (name, n_java, n_c)         # JNIEnv*, jclass + the Java parameters
    # the enumerations the plugin would instantiate implement the reference's interfaces by name
    enum = open(os.path.join(ROOT, "jni", PKG, "GpuTransformChunkEnumeration.java")).read()
    assert "implements TransformChunkEnumeration, AutoCloseable" in enum
    for method in ("originalChunkSize", "transformedChunkSize", "hasMoreElements", "nextElement", "close"):
        assert re.search(r"\b" + method + r"\s*\(", enum), method
    assert "readNBytes" not in enum and "channel.read(in)" in enum            # the stream lands in pinned memory, no byte[] bounce
    de = open(os.path.join(ROOT, "jni", PKG, "GpuDetransformChunkEnumeration.java")).read()
    assert "implements DetransformChunkEnumeration, AutoCloseable" in de and "Stream has fewer bytes than expected" in de
    for method in ("hasMoreElements", "nextElement", "close"):
        assert re.search(r"\b" + method + r"\s*\(", de), method
    cm = open(os.path.join(ROOT, "jni", "io/aiven/kafka/tieredstorage/fetch/gpu/GpuChunkManager.java")).read()
    assert "implements ChunkManager" in cm and "getChunks" in cm and "BytesRange.of(" in cm
    pool = open(os.path.join(ROOT, "jni", PKG, "PinnedPool.java")).read()
    assert "TsGpu.freePinned" in pool and "Cleaner" in pool                   # pinned memory is returned, also for leaked leases


def test_java_sources_reference_only_existing_reference_members():
    """The Java cannot be compiled without a JDK: at least every reference type / member the sources name must exist in
    the reference, whose declarations tests/golden/reference_vectors.json carries (java_api, transcribed with file:line)."""
    files = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_vectors.json")))["java_api"]["files"]
    ref = {f: "\n".join(e["declarations"]) for f, e in files.items()}
    chunk = ref["M/Chunk.java"]
    for field in ("transformedPosition", "transformedSize", "originalSize"):
        assert re.search(r"public final int " + field, chunk)
    assert "SecretKey dataKey();" in ref["M/manifest/SegmentEncryptionMetadata.java"]
    assert "InputStream getChunk(" in ref["M/fetch/ChunkManager.java"]
    assert "interface DetransformChunkEnumeration extends Enumeration<byte[]>" in ref["M/transform/DetransformChunkEnumeration.java"]
    assert "public static BytesRange of(final int from, final int to)" in ref["S/storage/BytesRange.java"]
