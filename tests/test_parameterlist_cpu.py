"""The ParameterList machinery of the drop-in boundary on the CPU: SimpleXMLParameterListReader
(src/utilities/ParELAG_SimpleXMLParameterListReader.cpp:55-380) and SolverLibrary::GetSolverFactory
(src/linalg/factories/ParELAG_SolverLibrary.cpp:36-67) through the C ABI, on a document that exercises the reader's rules
(compared with an independent parse by xml.etree)."""
import xml.etree.ElementTree as ET

import pytest

from parelag_b200 import api, capi


def fmt(typ, val):
    """the canonical form pe_api_parameterlist_dump prints"""
    if typ == "bool":
        return "true" if val.upper() == "TRUE" else "false"          # :223-236: "true" in any letter case
    if typ in ("int", "long", "long long", "unsigned long", "unsigned long long", "size_t", "char"):
        return str(int(val))
    if typ in ("double", "float", "long double"):
        return "%.17g" % float(val)
    if typ in ("vector(int)", "vector_int"):
        return " ".join(str(int(t)) for t in val.split())
    if typ in ("vector(double)", "vector_double"):
        return " ".join("%.17g" % float(t) for t in val.split())
    if typ == "list(string)":
        return ",".join(t.strip() for t in val.split(","))            # :272-286: comma separated, trimmed
    return val


def etree_dump(text):
    names = {"vector_int": "vector(int)", "vector_double": "vector(double)", "size_t": "unsigned long"}
    out = []

    def walk(node, prefix):
        for ch in node:
            if ch.tag == "ParameterList":
                walk(ch, prefix + ch.attrib["name"] + "/")
            elif ch.tag == "Parameter":
                t = ch.attrib["type"]
                out.append("%s%s\t%s\t%s" % (prefix, ch.attrib["name"], names.get(t, t), fmt(t, ch.attrib["value"])))
    walk(ET.fromstring(text), "")
    return sorted(out)


def test_reader_rules():
    doc = """<?xml version="1.0"?>
<!-- a comment with <tags> and = signs -->
<ParameterList name="Default">
  <Parameter name = "Type"   type="string" value="Hiptmair"/>
  <Parameter name="flag a" type="bool" value="True"/> <Parameter name="flag b" type="bool" value="TRUE"/>
  <Parameter name="flag c" type="bool" value="1"/>
  <Parameter name="solvers" type="list(string)"
             value="PCG-AMGe , GMRES with spaces,last"/>
  <ParameterList name="Sub list">
    <!--Parameter name="off" type="int" value="3"/-->
    <Parameter name="n" type="int" value="-7"/> <Parameter name="big" type="size_t" value="5000000000"/>
    <Parameter name="x" type="double" value="1e-6"/> <Parameter name="v" type="vector(int)" value="2 3"/>
    <Parameter name="w" type="vector_double" value="0.5 1.5e3"/> <Parameter name="l" type="long long" value="-9000000000"/>
    <ParameterList name="Empty"/>
  </ParameterList>
</ParameterList>"""
    got = api.parameterlist_dump(doc)
    assert got == sorted([
        "Type\tstring\tHiptmair", "flag a\tbool\ttrue", "flag b\tbool\ttrue", "flag c\tbool\tfalse",
        "solvers\tlist(string)\tPCG-AMGe,GMRES with spaces,last",
        "Sub list/n\tint\t-7", "Sub list/big\tunsigned long\t5000000000", "Sub list/x\tdouble\t9.9999999999999995e-07",
        "Sub list/v\tvector(int)\t2 3", "Sub list/w\tvector(double)\t0.5 1500", "Sub list/l\tlong long\t-9000000000"])
    assert got == etree_dump(doc)
    with pytest.raises(capi.PEError):
        api.parameterlist_dump('<ParameterList name="x"><Parameter name="a" type="quaternion" value="1"/></ParameterList>')
    with pytest.raises(capi.PEError):
        api.parameterlist_dump('<ParameterList name="x"><Parameter name="a" type="int" value=""/></ParameterList>')


def test_failed_factory_is_not_cached():
    """a factory whose initialisation fails (unknown nested type) must fail again when asked for directly"""
    lib = {"Outer": ("Krylov", {"Solver name": "PCG", "Preconditioner": "Inner"}), "Inner": ("BoomerAMG", {})}
    rep = dict((n, s) for n, t, s in api.library_factories(api.library_xml(lib)))
    assert rep["Inner"].startswith("error") and "BoomerAMG" in rep["Inner"]
    assert rep["Outer"].startswith("error") and "BoomerAMG" in rep["Outer"]


def test_block_gs_use_triangle_parameter():
    """ParELAG_Block2x2GaussSeidelSolverFactory.cpp:147-165: "Use triangle" = Lower | Upper in any letter case, else an error"""
    gs = ("Hypre", {"Type": "Gauss-Seidel"})
    for value, ok in (("Lower", True), ("upper", True), ("UPPER", True), ("diagonal", False)):
        lib = {"GS": gs, "B": ("Block GS", {"A00 Inverse": "GS", "A11 Inverse": "GS", "Use triangle": value})}
        rep = dict((n, s) for n, t, s in api.library_factories(api.library_xml(lib)))
        assert (rep["B"] == "ok") == ok, (value, rep["B"])
        if not ok:
            assert "Use triangle" in rep["B"]
