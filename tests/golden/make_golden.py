#!/usr/bin/env python
"""Writes the fixtures under tests/golden/.  Run from the repo root: `python tests/golden/make_golden.py`.

Two kinds of content:
  reference_vectors.json   golden vectors TRANSCRIBED from the reference's own tests (values only; each entry cites
                           the file:line it was read from, T = core/src/test/java/io/aiven/kafka/tieredstorage) plus the
                           public AES-256 GCM-specification / FIPS-197 known answers the AES path is pinned on, and the
                           declarations of the reference members the Java sources under jni/ use.
  libzstd_frames.json      frames GENERATED here by the oracle's libzstd (system libzstd, dlopen) from corpus.gen_chunk
                           inputs, at the level the reference uses (3) and at 1 / 19 for coverage, so that the decoder
                           parity tests do not depend on which libzstd the test box carries.  The reference is Java and
                           cannot run here (no JVM), so nothing in this file was produced by the reference itself.
The tests read these files; nothing under tests/golden/ is imported by the product.
"""
import base64
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))

REFERENCE_VECTORS = {
    "encoded_chunks": {
        "source": "T/manifest/index/ChunkIndexSerializationTest.java:39-74",
        "sizes": [10, 20, 30],
        "codec_hex": "000000030000000a01000a0000001e",
        "base64": "KLUv/SAPeQAAAAAAAwAAAAoBAAoAAAAe",
    },
    "chunk_index_json": {
        "source": "T/manifest/index/ChunkIndexSerializationTest.java:63-74",
        "fixed": {"args": [100, 250, 110, 30],
                  "json": '{"type":"fixed","originalChunkSize":100,"originalFileSize":250,"transformedChunkSize":110,"finalTransformedChunkSize":30}'},
        "variable": {"args": [100, 250, [10, 20, 30]],
                     "json": '{"type":"variable","originalChunkSize":100,"originalFileSize":250,"transformedChunks":"KLUv/SAPeQAAAAAAAwAAAAoBAAoAAAAe"}'},
    },
    "materialized_chunks": {
        "source": "T/manifest/index/ChunkIndexSerializationTest.java:93-97,118-122 (id, originalPosition, originalSize, transformedPosition, transformedSize)",
        "fixed": [[0, 0, 100, 0, 110], [1, 100, 100, 110, 110], [2, 200, 50, 220, 30]],
        "variable": [[0, 0, 100, 0, 10], [1, 100, 100, 10, 20], [2, 200, 50, 30, 30]],
    },
    "codec_bytes_per_value": {
        "source": "T/manifest/index/serde/ChunkSizesBinaryCodecTest.java:34-118 (values, expected bytes per delta)",
        "cases": [[[0, 1000, 2, 44002, 369], 2],
                  [[2147483647, 2147483646, 2147483645, 10], 1],
                  [[1, 2, 3, 2147483647], 1],
                  [[1, 265, 275, 285, 2147483647], 2],
                  [[1, 65545, 65555, 65565, 2147483647], 3],
                  [[1, 16777225, 16777235, 16777245, 2147483647], 4]],
    },
    "aes256_gcm_kats": {
        "source": "McGrew & Viega, The Galois/Counter Mode of Operation (GCM), Appendix B, test cases 13-16 (AES-256); public",
        "cases": [
            {"key": "00" * 32, "iv": "00" * 12, "aad": "", "pt": "", "ct": "", "tag": "530f8afbc74536b9a963b4f1c4cb738b"},
            {"key": "00" * 32, "iv": "00" * 12, "aad": "", "pt": "00" * 16, "ct": "cea7403d4d606b6e074ec5d3baf39d18",
             "tag": "d0d1c8a799996bf0265b98b5d48ab919"},
            {"key": "feffe9928665731c6d6a8f9467308308feffe9928665731c6d6a8f9467308308", "iv": "cafebabefacedbaddecaf888", "aad": "",
             "pt": "d9313225f88406e5a55909c5aff5269a86a7a9531534f7da2e4c303d8a318a721c3c0c95956809532fcf0e2449a6b525b16aedf5aa0de657ba637b391aafd255",
             "ct": "522dc1f099567d07f47f37a32a84427d643a8cdcbfe5c0c97598a2bd2555d1aa8cb08e48590dbb3da7b08b1056828838c5f61e6393ba7a0abcc9f662898015ad",
             "tag": "b094dac5d93471bdec1a502270e3cc6c"},
            {"key": "feffe9928665731c6d6a8f9467308308feffe9928665731c6d6a8f9467308308", "iv": "cafebabefacedbaddecaf888",
             "aad": "feedfacedeadbeeffeedfacedeadbeefabaddad2",
             "pt": "d9313225f88406e5a55909c5aff5269a86a7a9531534f7da2e4c303d8a318a721c3c0c95956809532fcf0e2449a6b525b16aedf5aa0de657ba637b39",
             "ct": "522dc1f099567d07f47f37a32a84427d643a8cdcbfe5c0c97598a2bd2555d1aa8cb08e48590dbb3da7b08b1056828838c5f61e6393ba7a0abcc9f662",
             "tag": "76fc6ece0f4e1768cddf8853bb2d551b"},
        ],
    },
    "aes256_block": {
        "source": "FIPS-197 Appendix C.3; public",
        "key": "000102030405060708090a0b0c0d0e0f101112131415161718191a1b1c1d1e1f",
        "pt": "00112233445566778899aabbccddeeff", "ct": "8ea2b7ca516745bfeafc49904b496089",
    },
    "java_api": {
        "source": "declarations of the reference types / members jni/ names, transcribed from the reference's main sources "
                  "(M = core/src/main/java/io/aiven/kafka/tieredstorage, S = storage/core/src/main/java/io/aiven/kafka/tieredstorage)",
        "files": {
            "M/Chunk.java": {"lines": "22-26", "declarations": [
                "public final int id;", "public final int originalPosition;", "public final int originalSize;",
                "public final int transformedPosition;", "public final int transformedSize;"]},
            "M/manifest/SegmentEncryptionMetadata.java": {"lines": "24", "declarations": ["SecretKey dataKey();"]},
            "M/fetch/ChunkManager.java": {"lines": "28", "declarations": ["InputStream getChunk(final ObjectKey objectKey,"]},
            "M/transform/DetransformChunkEnumeration.java": {"lines": "28", "declarations": [
                "public interface DetransformChunkEnumeration extends Enumeration<byte[]> {"]},
            "S/storage/BytesRange.java": {"lines": "100", "declarations": ["public static BytesRange of(final int from, final int to) {"]},
        },
    },
}


DENSE_CASES = (("K", 11, 300000, 131072), ("K", 12, 70001, 70001), ("R", 13, 40000, 40000), ("Z", 14, 70000, 32768),
               ("K", 15, 1 << 19, 1 << 19), ("K", 16, 8192 * 3 + 17, 8192))


def main():
    with open(os.path.join(HERE, "reference_vectors.json"), "w") as f:
        json.dump(REFERENCE_VECTORS, f, indent=1)
        f.write("\n")
    from oracle import oracle as ora
    import tsgpu
    from tsgpu import corpus
    frames = {"generator": "oracle (%s) via tests/golden/make_golden.py" % ora.lib().ora_zstd_version().decode(), "frames": []}
    for kind, seed, n, level in (("K", 1, 1, 3), ("K", 2, 300, 3), ("K", 3, 20000, 3), ("K", 4, 150000, 3), ("K", 5, 150000, 1),
                                 ("K", 6, 150000, 19), ("R", 7, 40000, 3), ("Z", 8, 70000, 3), ("K", 9, 400000, 3)):
        src = corpus.gen_chunk(kind, seed, 0, n)
        frame = ora.zstd_compress_level(src, level)
        frames["frames"].append({"kind": kind, "seed": seed, "n": n, "level": level,
                                 "sha256": hashlib.sha256(src.tobytes()).hexdigest(),
                                 "frame_b64": base64.b64encode(frame).decode()})
    with open(os.path.join(HERE, "libzstd_frames.json"), "w") as f:
        json.dump(frames, f, indent=1)
        f.write("\n")
    print("wrote", len(frames["frames"]), "frames,", sum(len(x["frame_b64"]) for x in frames["frames"]), "base64 bytes")
    # dense-mode frames of THIS library are a function of the input (DESIGN.md 4.2): digests of what the emulated kernels write,
    # so that (a) an unintended change of the compressed bytes shows up and (b) the B200 can be checked against the emulator
    import subprocess
    simt = os.path.join(ROOT, "tests", "simt", "libtsgpu_simt.so")
    subprocess.check_call(["make", "-s", "-C", ROOT, "tests/simt/libtsgpu_simt.so"])
    ctx = tsgpu.Context(max_chunk_bytes=1 << 19, max_batch=4, lib_path=simt)
    dense = {"generator": "the product's dense compressor (TSGPU_FLAG_ZSTD | TSGPU_FLAG_ZSTD_DENSE) under the test-only SIMT emulator, "
                          "tests/golden/make_golden.py", "cases": []}
    for kind, seed, n, cs in DENSE_CASES:
        src = corpus.gen_segment(kind, seed, n, cs)
        out, sizes = ctx.transform(tsgpu.FLAG_ZSTD | tsgpu.FLAG_ZSTD_DENSE, src, cs)
        dense["cases"].append({"kind": kind, "seed": seed, "n": n, "chunk_size": cs, "sizes": [int(x) for x in sizes],
                               "sha256": hashlib.sha256(out.tobytes()).hexdigest()})
    ctx.close()
    with open(os.path.join(HERE, "dense_frames.json"), "w") as f:
        json.dump(dense, f, indent=1)
        f.write("\n")
    print("wrote", len(dense["cases"]), "dense-frame digests")


if __name__ == "__main__":
    main()
