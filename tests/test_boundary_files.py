"""The non-code boundary files stay signature-compatible with the reference: its GRC descriptor signature and the
public declarations of its lib/baz_music_doa.h are stored in tests/golden/reference_source/surface.json
(tests/golden/make_reference_golden.py)."""
import json
import os
import re
import xml.etree.ElementTree as ET

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SURFACE = os.path.join(ROOT, "tests", "golden", "reference_source", "surface.json")


def reference_surface():
    with open(SURFACE) as f:
        return json.load(f)


def _sig(root):
    return (root.findtext("key"), root.findtext("import"), root.findtext("make"), root.findtext("callback"),
            [(p.findtext("key"), p.findtext("value"), p.findtext("type")) for p in root.findall("param")],
            [(s.findtext("name"), s.findtext("type"), s.findtext("vlen")) for s in root.findall("sink")],
            [(s.findtext("name"), s.findtext("type"), s.findtext("vlen"), s.findtext("optional")) for s in root.findall("source")])


def test_grc_descriptor_is_compatible_with_reference():
    b = ET.parse(os.path.join(ROOT, "grc", "baz_music_doa.xml")).getroot()
    assert json.loads(json.dumps(_sig(b))) == reference_surface()["grc_signature"]


def _decls(text):
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    return re.sub(r"\s+", " ", text)


def _norm(s):
    return re.sub(r"\s*([&*(),])\s*", r"\1", s)


# the declarations of the reference's lib/baz_music_doa.h a drop-in must keep
CPP_SURFACE = (
    "class baz_music_doa : public gr::sync_block",
    "typedef boost::shared_ptr<baz_music_doa> baz_music_doa_sptr;",
    "typedef std::vector<gr_complex> antenna_response_t;",
    "typedef std::vector<antenna_response_t> array_response_t;",
    "baz_music_doa_sptr baz_make_music_doa(unsigned int m, unsigned int n, unsigned int nsamples, const array_response_t& array_response, unsigned int resolution);",
    "int work(int noutput_items, gr_vector_const_void_star &input_items, gr_vector_void_star &output_items);",
    "void set_array_response(const array_response_t& array_response);",
)


def test_cpp_surface_matches_reference_header():
    ref = reference_surface()["cpp_declarations"]
    ours = _norm(_decls(open(os.path.join(ROOT, "lib", "baz_music_doa.h")).read()))
    for must in CPP_SURFACE:
        assert _norm(must) in ref, must
        assert _norm(must) in ours, must


def test_swig_fragment_keeps_python_name():
    s = open(os.path.join(ROOT, "swig", "baz_music_doa.i")).read()
    assert "GR_SWIG_BLOCK_MAGIC(baz,music_doa)" in s
    assert "std::vector<std::vector<gr_complex> >& array_response" in s
