"""Builds tests/golden/nvm_inputs_v1.npz and tests/golden/line3dpp_ref_fixture_v1.npz from the reference's test data
(run in the build container, where /root/reference exists and cv2 has an LSD):

    python tests/golden/make_nvm_inputs.py            # python tests/golden/make_nvm_inputs.py --sample: the reader fixture

nvm_inputs_v1.npz: what runLine3Dpp_vsfm hands to Line3D::addImage for testdata/vsfm_result.nvm
  (main_vsfm.cpp:143-310): per camera K (f, w/2, h/2), R (from the quaternion), t = -R C, median world-point depth,
  world-point id list; plus 2D segments detected like Line3D::detectLineSegments (line3D.cc:249-372): LSD_REFINE_ADV on
  the full-size grayscale image, keep length > 0.005*diag, longest 3000 first.  (cv2 4.x's LSD is not the LSD build the
  reference fixture was made with, so segment ids do not line up with the fixture; see SURVEY.md §4.)
line3dpp_ref_fixture_v1.npz: the 3D segments + 2D residuals of testdata/Line3D++_ref/*.txt (README.md:272-277 format),
  used for the statistical end-to-end comparison.
"""
import os
import sys

import numpy as np

REF = "/root/reference/testdata"
OUT = os.path.dirname(os.path.abspath(__file__))


def read_nvm(path):
    L = open(path).read().split("\n")
    ncam = int(L[2].split()[0])
    cams = []
    for i in range(ncam):
        p = L[3 + i].split()
        name, f = p[0], float(p[1])
        qw, qx, qy, qz = (float(x) for x in p[2:6])
        C = np.array([float(x) for x in p[6:9]])
        R = np.array([[1 - 2 * qy * qy - 2 * qz * qz, 2 * qx * qy - 2 * qz * qw, 2 * qx * qz + 2 * qy * qw],
                      [2 * qx * qy + 2 * qz * qw, 1 - 2 * qx * qx - 2 * qz * qz, 2 * qy * qz - 2 * qx * qw],
                      [2 * qx * qz - 2 * qy * qw, 2 * qy * qz + 2 * qx * qw, 1 - 2 * qx * qx - 2 * qy * qy]])
        cams.append(dict(name=os.path.basename(name), f=np.float32(f), R=R, C=C, t=-R @ C, dist=float(p[9])))
    npts = int(L[4 + ncam].split()[0])
    wps = [[] for _ in range(ncam)]
    depths = [[] for _ in range(ncam)]
    for i in range(npts):
        p = L[5 + ncam + i].split()
        pos = np.array([float(x) for x in p[0:3]])
        nv = int(p[6])
        for j in range(nv):
            cam = int(p[7 + 4 * j])
            wps[cam].append(i)
            depths[cam].append(np.float32(np.linalg.norm(pos - cams[cam]["C"])))
    return cams, wps, depths


def detect(gray, max_segments=3000):
    import cv2
    lsd = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV)
    det = lsd.detect(gray)[0].reshape(-1, 4).astype(np.float32)
    h, w = gray.shape
    diag = np.sqrt(np.float32(h * h) + np.float32(w * w))
    dx, dy = det[:, 0] - det[:, 2], det[:, 1] - det[:, 3]
    length = np.sqrt(dx * dx + dy * dy)
    keep = length > diag * np.float32(0.005)
    det, length = det[keep], length[keep]
    order = np.argsort(-length, kind="stable")[:max_segments]
    return det[order]


def read_fixture(path):
    segs, seg_line, res = [], [], []
    for li, line in enumerate(open(path)):
        p = line.split()
        if not p:
            continue
        n = int(p[0])
        for k in range(n):
            segs.append([float(x) for x in p[1 + 6 * k:7 + 6 * k]])
            seg_line.append(li)
        o = 1 + 6 * n
        m = int(p[o])
        for k in range(m):
            q = p[o + 1 + 6 * k:o + 7 + 6 * k]
            res.append((li, int(q[0]), int(q[1]), float(q[2]), float(q[3]), float(q[4]), float(q[5])))
    return np.array(segs), np.array(seg_line, np.int32), np.array(res)


def main():
    import cv2
    cams, wps, depths = read_nvm(os.path.join(REF, "vsfm_result.nvm"))
    g = {}
    V = len(cams)
    K = np.zeros((V, 3, 3)); R = np.zeros((V, 3, 3)); t = np.zeros((V, 3)); md = np.zeros(V, np.float32); wh = np.zeros((V, 2), np.int32)
    for i, c in enumerate(cams):
        img = cv2.imread(os.path.join(REF, c["name"]), cv2.IMREAD_GRAYSCALE)
        assert img is not None, c["name"]
        h, w = img.shape
        K[i] = [[c["f"], 0, np.float32(w) / np.float32(2)], [0, c["f"], np.float32(h) / np.float32(2)], [0, 0, 1]]
        if abs(c["dist"]) > 1e-12:        # main_vsfm.cpp:288-299 -> Line3D::undistortImage (line3D.cc:83-109), radial = (-d, 0, 0)
            dc = np.array([-np.float32(c["dist"]), 0, 0, 0, 0], np.float64)
            m1, m2 = cv2.initUndistortRectifyMap(K[i], dc, np.eye(3), K[i], (w, h), cv2.CV_32FC1)
            img = cv2.remap(img, m1, m2, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT)
        R[i], t[i], wh[i] = c["R"], c["t"], (w, h)
        d = np.sort(np.array(depths[i], np.float32))
        md[i] = d[len(d) // 2]
        s = detect(img)
        g[f"segs_{i}"] = s
        g[f"wps_{i}"] = np.array(wps[i], np.uint32)
        print(i, c["name"], w, h, "segments", len(s), "wps", len(wps[i]), "median depth", md[i], flush=True)
    g.update(K=K, R=R, t=t, median_depth=md, wh=wh, names=np.array([c["name"] for c in cams]))
    np.savez_compressed(os.path.join(OUT, "nvm_inputs_v1.npz"), **g)
    fx = os.path.join(REF, "Line3D++_ref", "Line3D++__W_FULL__N_10__sigmaP_2.5__sigmaA_10__epiOverlap_0.25__kNN_10__vis_3.txt")
    segs, seg_line, res = read_fixture(fx)
    print("fixture:", len(set(seg_line.tolist())), "lines", len(segs), "3D segments", len(res), "residuals")
    np.savez_compressed(os.path.join(OUT, "line3dpp_ref_fixture_v1.npz"), segs3d=segs, seg_line=seg_line, residuals=res)


def sample_nvm(npts=500):
    """vsfm_result_sample_v1.nvm.gz: testdata/vsfm_result.nvm with every camera line and its PLY trailer verbatim, but only a
    fixed, seeded sample of npts of its 3D points (lines verbatim, file order kept), for the reader test"""
    import gzip
    L = open(os.path.join(REF, "vsfm_result.nvm")).read().split("\n")
    ncam = int(L[2].split()[0])
    n = int(L[4 + ncam].split()[0])
    keep = np.sort(np.random.default_rng(0).choice(n, npts, replace=False))
    out = L[:4 + ncam] + [str(npts)] + [L[5 + ncam + i] for i in keep] + L[5 + ncam + n:]
    with gzip.open(os.path.join(OUT, "vsfm_result_sample_v1.nvm.gz"), "wt", compresslevel=9) as f:
        f.write("\n".join(out))


if __name__ == "__main__":
    sys.exit(sample_nvm() if "--sample" in sys.argv else main())
