#!/usr/bin/env python
"""Extracts a sample of the reference's HRIR sphere (resources/IRC_1003_C.bin) into tests/golden/irc_1003_c_sample.npz.

    python tests/golden/extract_hrir_sample.py <web-audio-api-rs checkout>

The whole sphere is 755 KB of float32 responses that do not compress.  The sample keeps what the tests read from it:
  - the complete geometry (sample rate, tap count, vertex positions, triangle faces), bit for bit: the sphere lookup
    (library vs oracle) walks all of it;
  - the left / right responses of the vertices of every face around the vertex at +x, where the HRTF panner of
    src/node/panner.rs:1225-1269 test_hrtf looks (a source at x = 1 in front of the default listener).  Rendering that
    test with the sample gives the same bits as with the whole sphere at 44.1 and 48 kHz.
The responses of all other vertices are left out; tests/test_oracle_kat.py puts zeros in their place.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import graphs as G  # noqa: E402

OUT = os.path.join(HERE, "irc_1003_c_sample.npz")


def main():
    data = open(os.path.join(sys.argv[1], "resources", "IRC_1003_C.bin"), "rb").read()
    sr, pos, faces, left, right = G.parse_hrir_sphere(data)
    centre = int(np.argmax(pos[:, 0]))
    kept = np.unique(faces[(faces == centre).any(axis=1)]).astype(np.uint32)
    np.savez_compressed(OUT, sample_rate=np.uint32(sr), positions=pos, faces=faces, kept=kept, left=left[kept], right=right[kept])
    print(f"{OUT}: {len(pos)} vertices, {len(faces)} faces, responses of {len(kept)} vertices ({os.path.getsize(OUT)} bytes)")


if __name__ == "__main__":
    main()
