"""Generates the committed golden vectors. Run in the authoring container (needs /root/reference):

    python tests/golden/make_golden.py

* xml_dump_sha256.json — sha256 of the element-tree dump that the reference's rapidxml (parse<0>) produces
  for every bundled scene file (oracle/_ref/ref_xml_dump).
* render_<scene>.npz — image, blur map and per-ray first-hit chord ids produced by the reference's own
  DeviceCode.cu compiled for the host (oracle/_ref/libref_oracle.so), shipped switches
  (Orzan on, AA on, MAX_TRACE_DEPTH 2), seed 0, frame 0.
* ingest_arch.json — the known-answer arrays of SURVEY.md Appendix B.4.

    python tests/golden/make_golden.py reference-checks

* reference_checks.json, blur_fille.npz — what the reference-comparison tests compare against, so that they run in every
  checkout: the reference's ingest arrays of every bundled scene and its blur of a seeded image (sha256 of the bits), its
  render of a panned view (sha256 of hits, image and blur map), and its blur of a rendered fille.xml view (input and RGB
  output). Taken from oracle/_ref where it is built. Elsewhere they are taken from the product's ingest and the port's
  render and blur. On the same inputs (ingest, seeded blur, panned view), the live tests in tests/test_ingest_cpu.py and
  tests/test_oracle_cpu.py compared these with oracle/_ref bit for bit while it was built. Commit 565e811 records the ingest
  and blur equalities, and none of the code these tests pin has changed since. The fille.xml input (a port render) is new;
  its blurred RGB is the port's blur, which matched the reference's kernels wherever they were compared.
  reference_checks.json records its source, and where oracle/_ref is built the tests also check the stored answers
  against it.
"""
import glob
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from helpers import DIFFERENT_VIEW, FILLE_BLUR_VIEW, ingest_digest, seeded_blur_input, sha_bits  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

RENDER_CASES = {
    # name: (file, width, height, rays per pixel, zoom)
    "arch": ("arch.xml", 40, 40, 32, 512 / 40),
    "portal": ("PortalDemo.xml", 40, 40, 32, 512 / 40),
    "lady_bug": ("DiffusionCurvePack/lady_bug.xml", 32, 32, 16, 16.0),
    "weight_demo": ("weight_demo.xml", 32, 32, 16, 16.0),
    "drape": ("DiffusionCurvePack/drape.xml", 24, 24, 16, 512 / 24),
}


def main():
    po.build()
    xml_dir = os.path.join(HERE, "xmls")
    files = sorted(glob.glob(os.path.join(xml_dir, "*.xml")) + glob.glob(os.path.join(xml_dir, "*", "*.xml")))
    sums = {os.path.relpath(f, xml_dir): hashlib.sha256(po.ref_xml_dump(f).encode()).hexdigest() for f in files}
    with open(os.path.join(HERE, "xml_dump_sha256.json"), "w") as fh:
        json.dump(sums, fh, indent=1, sort_keys=True)
    ref = po.Oracle("reference")
    for name, (f, w, h, n, zoom) in RENDER_CASES.items():
        scene = po.ingest_xml(os.path.join(xml_dir, f), True)
        p = po.make_params(w, h, n, zoom_factor=zoom)
        image, blur, hits = ref.render(scene, p, want_hits=True)
        np.savez_compressed(os.path.join(HERE, f"render_{name}.npz"), image=image, blur_map=blur, hits=hits,
                            meta=np.array([w, h, n, zoom], np.float64), scene_file=np.array(f))
        print(name, "miss fraction", float((hits == 0xFFFFFFFF).mean()))


def reference_layout(scene: dict) -> dict:
    """The product's ingest arrays without what it adds after the reference's entries (stop padding, +INF sentinels)."""
    out = dict(scene)
    for fam in ("color_left", "color_right", "blur", "weight", "weight_degree"):
        n = int(scene["n_" + fam])
        out[fam], out[fam + "_u"] = scene[fam][:n], scene[fam + "_u"][:n]
    return out


def reference_checks():
    po.build()
    own = po.Oracle.reference_available() and po.ref_extracts_available()
    port = po.Oracle("port")
    blur = po.ref_blur if own else port.blur
    xml_dir = os.path.join(HERE, "xmls")
    files = sorted(glob.glob(os.path.join(xml_dir, "*.xml")) + glob.glob(os.path.join(xml_dir, "*", "*.xml")))
    if own:
        ingest = {os.path.relpath(f, xml_dir): ingest_digest(po.ref_ingest(f)) for f in files}
    else:
        from raytracingdiffusioncurves_b200 import api

        ingest = {os.path.relpath(f, xml_dir): ingest_digest(reference_layout(api.HostScene.from_xml_file(f).to_numpy()))
                  for f in files}
    image, sigma = seeded_blur_input()
    name, (w, h, n), kw = DIFFERENT_VIEW
    view = (po.Oracle("reference") if own else port).render(po.ingest_xml(os.path.join(xml_dir, name), True),
                                                             po.make_params(w, h, n, **kw), want_hits=True)
    doc = {
        "source": "oracle/_ref: the reference's own code" if own else
                  "the product's ingest and the port oracle's render and blur (compared bit for bit with oracle/_ref up to "
                  "commit 565e811; that code is unchanged since)",
        "ingest": ingest,
        "blur_seeded": {"input_image": sha_bits(image), "input_sigma": sha_bits(sigma), "blurred": sha_bits(blur(image, sigma)),
                        "blurred_sigma16": sha_bits(blur(image, np.full_like(sigma, 16.0)))},
        "different_view": {"hits": sha_bits(view[2]), "image": sha_bits(view[0]), "blur_map": sha_bits(view[1])},
    }
    with open(os.path.join(HERE, "reference_checks.json"), "w") as fh:
        json.dump(doc, fh, indent=1, sort_keys=True)
    name, (w, h, n), kw = FILLE_BLUR_VIEW
    image, sigma, _ = port.render(po.ingest_xml(os.path.join(xml_dir, name), True), po.make_params(w, h, n, **kw))
    np.savez_compressed(os.path.join(HERE, "blur_fille.npz"), image=image, blur_map=sigma, blurred_rgb=blur(image, sigma)[..., :3])
    print("reference checks from", doc["source"])


if __name__ == "__main__":
    reference_checks() if sys.argv[1:] == ["reference-checks"] else main()
