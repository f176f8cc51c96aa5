"""Fixtures that stand in for the reference tree in the checkpoint and parameter-inventory tests.

    python tests/golden/make_golden_checkpoints.py <reference root>

  checkpoint_layout.npz     The two shipped MXNet checkpoints the tests read (weights/dbbSep30-1206_1000000.params,
                            MaskFlownet-S; weights/5adNov03-0005_1000000.params, the cascade) without their weight data:
                            every other byte of the file verbatim (list header, per-array headers, name table), the place
                            and size of each array's data, and 16 seeded weight values per array.  rebuild_checkpoint()
                            writes a file with exactly the original byte layout whose arrays are zero except at the
                            sampled elements, which hold the shipped values.  (The originals are 42 and 83 MB.)
  ref_param_inventory.json  Name and shape of every parameter the reference's network/MaskFlownet.py creates for
                            MaskFlownet_S and MaskFlownet (imported unchanged through maskflownet_b200.mx, shapes
                            materialised by one forward pass on the oracle operators), in creation order.
"""
import json
import os
import struct
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LAYOUT = os.path.join(HERE, "checkpoint_layout.npz")
INVENTORY = os.path.join(HERE, "ref_param_inventory.json")
CHECKPOINT_S = "dbbSep30-1206_1000000"
CHECKPOINT_CASCADE = "5adNov03-0005_1000000"
SAMPLES_PER_ARRAY = 16


def rebuild_checkpoint(stem: str, directory: str) -> str:
    """Write <directory>/<stem>.params from checkpoint_layout.npz; returns its path."""
    d = np.load(LAYOUT)
    skel, holes = d[stem + "/skeleton"].tobytes(), d[stem + "/holes"]
    parts, prev = [], 0
    for at, n in holes:
        parts += [skel[prev:at], bytes(int(n))]
        prev = int(at)
    parts.append(skel[prev:])
    buf = bytearray(b"".join(parts))
    data_off = holes[:, 0] + np.concatenate([[0], np.cumsum(holes[:-1, 1])])     # array starts in the full file
    pos = data_off[d[stem + "/sample_array"]] + 4 * d[stem + "/sample_index"]
    u8 = np.frombuffer(buf, dtype=np.uint8)
    u8[pos[:, None] + np.arange(4)] = d[stem + "/sample_value"].astype("<f4").view(np.uint8).reshape(-1, 4)
    path = os.path.join(directory, stem + ".params")
    with open(path, "wb") as f:
        f.write(buf)
    return path


def shipped_samples(stem: str):
    """(array position in the file, flat element index, shipped float32 value) of every stored sample."""
    d = np.load(LAYOUT)
    return list(zip(d[stem + "/sample_array"].tolist(), d[stem + "/sample_index"].tolist(),
                    d[stem + "/sample_value"].tolist()))


def _layout(path: str, rng):
    buf = open(path, "rb").read()
    off = 24
    magic, _, n = struct.unpack_from("<QQQ", buf, 0)
    assert magic == 0x112
    skel, holes, prev, s_arr, s_idx, s_val = [], [], 0, [], [], []
    for a in range(n):
        nd_magic, stype, ndim = struct.unpack_from("<IiI", buf, off)
        assert nd_magic == 0xF993FAC9 and stype == 0
        dims = struct.unpack_from(f"<{ndim}q", buf, off + 12)
        dtype_flag = struct.unpack_from("<i", buf, off + 12 + 8 * ndim + 8)[0]
        assert dtype_flag == 0                                  # float32
        off += 12 + 8 * ndim + 12
        cnt = int(np.prod(dims))
        skel.append(buf[prev:off])
        holes.append((sum(map(len, skel)), 4 * cnt))
        idx = np.sort(rng.choice(cnt, size=min(SAMPLES_PER_ARRAY, cnt), replace=False))
        s_arr += [a] * len(idx)
        s_idx += idx.tolist()
        s_val += np.frombuffer(buf, dtype="<f4", count=cnt, offset=off)[idx].tolist()
        off += 4 * cnt
        prev = off
    skel.append(buf[prev:])
    return {"skeleton": np.frombuffer(b"".join(skel), dtype=np.uint8), "holes": np.array(holes, dtype=np.int64),
            "sample_array": np.array(s_arr, dtype=np.int64), "sample_index": np.array(s_idx, dtype=np.int64),
            "sample_value": np.array(s_val, dtype=np.float32)}


def main(reference_root: str):
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    sys.path.insert(0, HERE)
    from make_golden import load_reference_on_oracle, seeded_images
    from maskflownet_b200 import mx, params

    rng = np.random.default_rng(0)
    out = {}
    for stem in (CHECKPOINT_S, CHECKPOINT_CASCADE):
        src = os.path.join(reference_root, "weights", stem + ".params")
        for k, v in _layout(src, rng).items():
            out[f"{stem}/{k}"] = v
    np.savez_compressed(LAYOUT, **out)
    # the rebuilt file parses to the original's names and shapes, and carries the shipped values where they were sampled
    for stem in (CHECKPOINT_S, CHECKPOINT_CASCADE):
        orig = params.read_params(os.path.join(reference_root, "weights", stem + ".params"))
        with tempfile.TemporaryDirectory() as tmp:
            rebuilt = params.read_params(rebuild_checkpoint(stem, tmp))
        assert [(k, v.shape) for k, v in orig.items()] == [(k, v.shape) for k, v in rebuilt.items()]
        names = list(orig)
        for a, i, v in shipped_samples(stem):
            assert orig[names[a]].flat[i] == v == rebuilt[names[a]].flat[i]

    ref = load_reference_on_oracle(reference_root)
    im1, im2 = seeded_images()
    inventory = {}
    for cls in ("MaskFlownet_S", "MaskFlownet"):
        net = getattr(ref, cls)(config=mx.Reader({}))
        net.initialize(seed=0, device="cpu")
        with torch.no_grad():
            net(mx.nd.NDArray(im1), mx.nd.NDArray(im2))         # materialises the deferred shapes
        inventory[cls] = [[name, list(p.shape)] for name, p in net.collect_params().items()]
    with open(INVENTORY, "w") as f:                             # one parameter per line
        f.write("{\n" + ",\n".join(f"{json.dumps(cls)}: [\n" + ",\n".join(json.dumps(e) for e in entries) + "\n]"
                                   for cls, entries in inventory.items()) + "\n}\n")
    print("wrote", LAYOUT, "and", INVENTORY)


if __name__ == "__main__":
    main(sys.argv[1])
