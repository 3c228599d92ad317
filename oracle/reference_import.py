"""ORACLE helper: import the reference's own wiring files UNMODIFIED from a checkout of the reference (read-only) on top
of the diffusers stand-in.  The checkout is named by T2V_REFERENCE_ROOT; the golden generators under tests/golden/ need
it, the tests compare with the fixtures those generators stored."""
import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get("T2V_REFERENCE_ROOT", "")
_STANDIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "diffusers_standin")


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "unet_3d_condition.py"))


def import_reference_unet():
    """Returns the reference's UNet3DConditionModel class (its module is registered as `_refpkg.models...`)."""
    if not reference_available():
        raise RuntimeError("reference sources not present")
    try:
        import diffusers  # noqa: F401  (a real install wins if it ever exists)
    except ImportError:
        if _STANDIN not in sys.path:
            sys.path.insert(0, _STANDIN)
    # Load reference `models` as an isolated package so it cannot shadow / be shadowed by the product's `models`.
    import importlib.util
    pkg_name = "_t2v_reference_models"
    if pkg_name not in sys.modules:
        spec = importlib.util.spec_from_file_location(
            pkg_name, os.path.join(REFERENCE_ROOT, "models", "__init__.py"),
            submodule_search_locations=[os.path.join(REFERENCE_ROOT, "models")])
        if spec is None or not os.path.exists(os.path.join(REFERENCE_ROOT, "models", "__init__.py")):
            import types
            pkg = types.ModuleType(pkg_name)
            pkg.__path__ = [os.path.join(REFERENCE_ROOT, "models")]
            sys.modules[pkg_name] = pkg
        else:
            pkg = importlib.util.module_from_spec(spec)
            sys.modules[pkg_name] = pkg
            spec.loader.exec_module(pkg)
    mod = importlib.import_module(pkg_name + ".unet_3d_condition")
    return mod.UNet3DConditionModel
