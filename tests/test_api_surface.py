"""Drop-in check of the Python boundary (SURVEY.md section 8b-i): every class, method, property and module-level function
the reference defines in pilco/ and safe_pilco_extension/ must exist here under the same import path with the same
leading positional parameters.  The reference's surface is stored in tests/golden/api_surface.json (read from its
sources with ``ast`` by tests/golden/make_api_surface.py)."""
import importlib
import inspect
import json
import os

SURFACE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "api_surface.json")


def test_public_surface_matches_reference():
    import pilco  # noqa: F401  (installs the alias modules)
    checked, problems = 0, []
    for modname, ref in json.load(open(SURFACE)).items():
        mod = importlib.import_module(modname)
        for name in ref["functions"]:
            checked += 1
            if not hasattr(mod, name):
                problems.append("missing function %s.%s" % (modname, name))
        for clsname, methods in ref["classes"].items():
            cls = getattr(mod, clsname, None)
            if cls is None:
                problems.append("missing class %s.%s" % (modname, clsname))
                continue
            for name, ref_args in methods:
                checked += 1
                if not hasattr(cls, name):
                    problems.append("missing %s.%s.%s" % (modname, clsname, name))
                    continue
                static = inspect.getattr_static(cls, name)
                if isinstance(static, property):
                    continue
                our_args = list(inspect.signature(getattr(cls, name)).parameters)
                if our_args[:len(ref_args)] != ref_args:
                    problems.append("signature %s.%s.%s: reference %s, here %s" % (modname, clsname, name, ref_args, our_args))
    assert not problems, "\n".join(problems)
    assert checked >= 50
