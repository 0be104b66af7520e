#!/usr/bin/env python
"""Record what the UNMODIFIED reference engine does with the files of tests/test_gpu_ref_interop.py into a JSON fixture.

Needs a CUDA device and oracle/_ref/storage_offload_ref.so (built by oracle/ref_build/build_ref.py from the reference
sources, llm-d/llm-d-kv-cache @ 82d31d1):
    python tests/golden/make_ref_interop.py [OUT.json]
For every file the reference writes (CPU path, gds_mode "disabled") it records the file size, where the payload starts
(found in the file, not taken from the oracle) and the SHA-256 of the payload bytes.  It also checks that the reference
restores every page from files written by this project's engine and from the oracle's file image with non-zero filler
outside the payload.  Only these facts are stored; the bytes are re-created by the test from the same seed.
"""
import hashlib
import importlib
import importlib.util
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import offload_oracle as oo  # noqa: E402
from tests.test_gpu_ref_interop import FRAG, T, interop_case  # noqa: E402

SO = os.path.join(ROOT, "oracle", "_ref", "storage_offload_ref.so")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_interop_golden.json")


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def drain(eng, job):
    t0 = time.time()
    while time.time() - t0 < 30:
        for j, ok in eng.get_finished():
            if j == job:
                return ok
        time.sleep(0.001)
    raise TimeoutError(job)


def restores(torch, eng_cls, src, files, ids, bpf):
    dst = [torch.zeros_like(t) for t in src]
    eng = eng_cls(2, bpf, dst, 1, "disabled", 0.0)
    eng.async_load_gpu_blocks(2, files, ids)
    assert drain(eng, 2)
    torch.cuda.synchronize()
    ok = all(torch.equal(d[b], s[b]) for d, s in zip(dst, src) for blk in ids for b in blk)
    del eng
    return ok


def main(out_path: str) -> None:
    import torch
    kvb = importlib.import_module("llm-d-kv-cache_b200")
    spec = importlib.util.spec_from_file_location("storage_offload_ref", SO)
    ref_mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_mod)
    tmp = tempfile.mkdtemp(prefix="kvb-ref-interop-")
    rec = {"_source": "llm-d/llm-d-kv-cache@82d31d1 StorageOffloadEngine (kv_connectors/llmd_fs_backend/csrc/storage), "
                      "CPU path, recorded on an NVIDIA B200 by tests/golden/make_ref_interop.py",
           "shape": {"tensors": T, "fragment_bytes": FRAG}}
    try:
        for bpf in (1, 4):
            src_np, ids = interop_case(bpf)
            rec["source_sha256"] = sha(src_np)
            src = [torch.from_numpy(s).cuda().view(torch.int8) for s in src_np]
            ref = ref_mod.StorageOffloadEngine(4, bpf, src, 3, "disabled", 0.0)
            f_ref = [f"{tmp}/{bpf}/ref/{i}.bin" for i in range(len(ids))]
            ref.async_store_gpu_blocks(1, f_ref, ids)
            assert drain(ref, 1)
            del ref
            files = []
            for f, blk in zip(f_ref, ids):
                img = np.fromfile(f, dtype=np.uint8)
                payload = oo.pack_blocks(list(src_np), blk)
                off = img.tobytes().find(payload[:FRAG].tobytes())
                assert off >= 0 and np.array_equal(img[off:off + payload.size], payload), f
                files.append({"blocks": blk, "size": int(img.size), "payload_offset": int(off),
                              "payload_bytes": int(payload.size), "payload_sha256": sha(img[off:off + payload.size])})
            ours = kvb.engine.StorageOffloadEngine(4, bpf, src, 3, "disabled", 0.0)
            f_our = [f"{tmp}/{bpf}/ours/{i}.bin" for i in range(len(ids))]
            assert ours.async_store_gpu_blocks(1, f_our, ids)
            assert drain(ours, 1)
            ours.shutdown()
            f_img = []
            for i, blk in enumerate(ids):
                f_img.append(f"{tmp}/{bpf}/image_{i}.bin")
                oo.file_image(list(src_np), blk, bpf, fill=0xA5).tofile(f_img[-1])
            rec[str(bpf)] = {
                "files": files,
                "reference_restores_files_of_this_engine": restores(torch, ref_mod.StorageOffloadEngine, src, f_our, ids,
                                                                    bpf),
                "reference_restores_oracle_image_with_filler": restores(torch, ref_mod.StorageOffloadEngine, src, f_img,
                                                                        ids, bpf),
            }
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else OUT)
