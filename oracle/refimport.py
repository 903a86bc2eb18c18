"""TEST INFRASTRUCTURE ONLY — loader for the *real* reference modules.

Works only where ``GFC_REFERENCE_ROOT`` names a checkout of the original project.
It is used by ``oracle/make_golden.py`` (to generate ``tests/golden/*.npz``) and
by the few CPU tests that run the reference's code live; without a checkout they
skip, and the goldens stand in for it.  Nothing in the product package may import
this file.

The reference's ``utils/__init__.py`` eagerly imports every sibling (matplotlib,
easydict … are absent here), so the packages are pre-seeded with empty
``ModuleType`` stubs whose ``__path__`` points at the reference directories.
"""
import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("GFC_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "utils", "graphUtils", "graphML.py"))


def _stub_pkg(name: str, path: str) -> None:
    if name in sys.modules and getattr(sys.modules[name], "__gfc_stub__", False):
        return
    m = types.ModuleType(name)
    m.__path__ = [path]
    m.__gfc_stub__ = True
    sys.modules[name] = m


def graphml():
    """reference ``utils/graphUtils/graphML.py`` (GraphFilterBatch :2369, BatchLSIGF :2273)."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    _stub_pkg("utils", os.path.join(REF_ROOT, "utils"))
    _stub_pkg("utils.graphUtils", os.path.join(REF_ROOT, "utils", "graphUtils"))
    return importlib.import_module("utils.graphUtils.graphML")


def graphtools():
    graphml()
    return importlib.import_module("utils.graphUtils.graphTools")


def scene_read_adj(pos_xy, max_range):
    """Run the reference ``Scene.readADjMatrix`` (scene.py:140-154) unbound on
    python-float positions ``pos_xy[N][2]``; returns float array ``[1, N*N]``."""
    if not available():
        raise RuntimeError("reference tree not present")
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    cwd = os.getcwd()
    try:
        os.chdir(REF_ROOT)  # sim.py loads remoteApi.so relative to cwd
        scene = importlib.import_module("scene")
    finally:
        os.chdir(cwd)
    robots = [types.SimpleNamespace(xi=types.SimpleNamespace(x=float(p[0]), y=float(p[1])))
              for p in pos_xy]
    fake_self = types.SimpleNamespace(robots=robots)
    return scene.Scene.readADjMatrix(fake_self, max_range)


def fixed_radius_gso(agent_pos, radius, zero_tol=1e-9):
    """Run the reference ``multiRobotSim.computeAdjacencyMatrix_fixedCommRadius``
    (utils/multirobotsim_dcenlocal.py:291-317) unbound.  ``agent_pos`` is
    ``[1, N, 2]`` float64.  Returns (S [1,N,N] float64, connected bool)."""
    graphml()
    _stub_pkg("dataloader", os.path.join(REF_ROOT, "dataloader"))
    if "dataloader.statetransformer" not in sys.modules:
        st = types.ModuleType("dataloader.statetransformer")
        st.AgentState = object
        sys.modules["dataloader.statetransformer"] = st
    if "utils.multipathvisualizerCombine" not in sys.modules:
        mv = types.ModuleType("utils.multipathvisualizerCombine")
        mv.DrawpathCombine = object
        sys.modules["utils.multipathvisualizerCombine"] = mv
    mod = importlib.import_module("utils.multirobotsim_dcenlocal")
    fake_self = types.SimpleNamespace(communicationRadius=radius, zeroTolerance=zero_tol)
    W, _r, conn = mod.multiRobotSim.computeAdjacencyMatrix_fixedCommRadius(
        fake_self, 0, agent_pos, radius)
    return W, conn


def decentral_planner_net(gml_module=None):
    """The reference policy class ``DecentralPlannerNet`` (graphs/models/suhaas_model.py:12-259).

    With ``gml_module`` the reference file is executed with ITS OWN ``import utils.graphUtils.graphML as gml``
    resolving to that module instead — the one-line swap of INTEGRATION.md §1 — so the returned class is the
    unmodified reference model wired to the drop-in layer (``suhaas_model.py:114``)."""
    ref_gml = graphml()
    _stub_pkg("graphs", os.path.join(REF_ROOT, "graphs"))
    _stub_pkg("graphs.models", os.path.join(REF_ROOT, "graphs", "models"))
    if "torchsummaryX" not in sys.modules:
        ts = types.ModuleType("torchsummaryX")
        ts.summary = lambda *a, **k: None
        sys.modules["torchsummaryX"] = ts
    importlib.import_module("graphs.weights_initializer")
    path = os.path.join(REF_ROOT, "graphs", "models", "suhaas_model.py")
    name = "graphs.models.suhaas_model" + ("" if gml_module is None else "__gfc_swapped")
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    pkg = sys.modules["utils.graphUtils"]
    saved_mod, saved_attr = sys.modules["utils.graphUtils.graphML"], getattr(pkg, "graphML", None)
    try:
        if gml_module is not None:   # `import a.b.c as x` binds sys.modules / the parent package attribute
            sys.modules["utils.graphUtils.graphML"] = gml_module
            pkg.graphML = gml_module
        spec.loader.exec_module(mod)
    finally:
        sys.modules["utils.graphUtils.graphML"] = saved_mod
        pkg.graphML = saved_attr if saved_attr is not None else ref_gml
    return mod.DecentralPlannerNet
