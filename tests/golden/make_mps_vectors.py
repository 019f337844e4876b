"""Extracts the reference's own MPS-limit test table into tests/golden/mps_limits.json.

Source: api/nvidia.com/resource/gpu/v1alpha1/sharing_test.go:37-149 of NVIDIA/k8s-dra-driver
(TestMpsPerDevicePinnedMemoryLimitNormalize, 14 table cases).  The tests read only the JSON, so they need no
checkout of that project:

  python tests/golden/make_mps_vectors.py <k8s-dra-driver checkout>
"""
import json
import os
import re
import sys

SRC = os.path.join("api", "nvidia.com", "resource", "gpu", "v1alpha1", "sharing_test.go")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mps_limits.json")


def main(reference_root):
    text = open(os.path.join(reference_root, SRC)).read()
    body = text[text.index("testCases := []struct"):text.index("for _, tc := range testCases")]
    body = body[body.index("}{") + 2:]
    cases = []
    # split on top-level "{ description:" blocks
    for blk in re.split(r"\n\t\t\{\n", "\n" + body)[1:]:
        d = re.search(r'description:\s*"([^"]*)"', blk).group(1)
        uu = re.search(r"uuids:\s*\[\]string\{([^}]*)\}", blk)
        uuids = re.findall(r'"([^"]*)"', uu.group(1)) if uu else []
        ml = re.search(r'memoryLimit:\s*ptr\(resource\.MustParse\("([^"]*)"\)\)', blk)
        pd = re.search(r"perDeviceMemoryLimit:\s*configapi\.MpsPerDevicePinnedMemoryLimit\{(.*?)\n\t\t\t\}", blk, re.S)
        per = dict(re.findall(r'"([^"]*)":\s*resource\.MustParse\("([^"]*)"\)', pd.group(1))) if pd else None
        er = re.search(r"expectedError:\s*configapi\.(\w+)", blk)
        el = re.search(r"expectedLimits:\s*map\[string\]string\{(.*?)\}", blk, re.S)
        limits = dict(re.findall(r'"([^"]*)":\s*"([^"]*)"', el.group(1))) if el else None
        cases.append({"description": d, "uuids": uuids, "memoryLimit": ml.group(1) if ml else None,
                      "perDeviceMemoryLimit": per, "expectedError": er.group(1) if er else None,
                      "expectedLimits": limits})
    assert len(cases) == 14, len(cases)
    json.dump({"source": "api/nvidia.com/resource/gpu/v1alpha1/sharing_test.go:37-149", "cases": cases},
              open(OUT, "w"), indent=1)
    print(f"wrote {OUT}: {len(cases)} cases")


if __name__ == "__main__":
    sys.exit(main(sys.argv[1]))
