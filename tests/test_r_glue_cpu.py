"""R is not installed in this image, so the .C() glue under R/ cannot be executed here.  This is a static check instead:
every .C("nngp_...") call names an exported ABI function and passes exactly as many arguments as the C prototype in
include/nngp_b200.h has parameters, named and ordered like them, with `status` last (.C() matches by position: a wrong
count or order corrupts memory at run time in R), and of the right KIND: .C() hands a double vector over as double *, an integer
vector as int *, and a character vector as char ** (never char *).  The patch for mcmc_nngp_initialize.R must apply to the
reference's lines it changes (tests/golden/mcmc_nngp_initialize_excerpt.R), and the .Call glue must compile against the R API declarations it uses."""
import os
import re
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def prototypes():
    src = open(os.path.join(ROOT, "include", "nngp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for name, args in re.findall(r"^void\s+(nngp_\w+)\s*\((.*?)\)\s*;", src, flags=re.M | re.S):
        params = [a.strip() for a in args.replace("\n", " ").split(",") if a.strip() and a.strip() != "void"]
        protos[name] = [re.sub(r".*[\s\*]", "", p) for p in params]
    return protos


def prototype_kinds():
    """name -> [kind per parameter]: "int", "double", "char**" (what .C() can pass) or "other" (char *, void **: not bindable with .C())"""
    src = open(os.path.join(ROOT, "include", "nngp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    kinds = {}
    for name, args in re.findall(r"^void\s+(nngp_\w+)\s*\((.*?)\)\s*;", src, flags=re.M | re.S):
        out = []
        for p in [a.strip() for a in args.replace("\n", " ").split(",") if a.strip() and a.strip() != "void"]:
            ty = re.sub(r"\w+$", "", p).replace("const", "").replace(" ", "")
            out.append({"int*": "int", "double*": "double", "char**": "char**"}.get(ty, "other"))
        kinds[name] = out
    return kinds


def r_kind(expr):
    """kind of an R argument expression as .C() will see it, or None when it cannot be told statically"""
    e = expr.strip()
    m = re.match(r"if\s*\(", e)
    if m:   # if(cond) a else b: both branches must agree
        depth, i = 1, m.end()
        while depth:
            depth += {"(": 1, ")": -1}.get(e[i], 0)
            i += 1
        a, _, b = e[i:].partition(" else ")
        ka, kb = r_kind(a), r_kind(b)
        return ka if ka == kb else None
    if re.match(r"(as\.double|double)\(", e) or re.fullmatch(r"-?\d+\.\d*", e):
        return "double"
    if re.match(r"(as\.integer|integer|length|nrow|ncol)\(", e) or re.fullmatch(r"-?\d+L", e):
        return "int"
    if re.match(r"(strrep|paste|paste0|character)\(", e) or re.fullmatch(r"\".*\"", e):
        return "char**"
    return None


def split_top_level(s):
    out, depth, cur, quote = [], 0, "", None
    for ch in s:
        if quote:
            cur += ch
            if ch == quote:
                quote = None
            continue
        if ch in "\"'":
            quote = ch
            cur += ch
        elif ch in "([{":
            depth += 1
            cur += ch
        elif ch in ")]}":
            depth -= 1
            cur += ch
        elif ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur.strip())
    return out


def dot_c_calls(text):
    calls = []
    for mobj in re.finditer(r"\.C\(", text):
        i, depth = mobj.end(), 1
        while depth:
            depth += {"(": 1, ")": -1}.get(text[i], 0)
            i += 1
        args = split_top_level(text[mobj.end():i - 1])
        name = args[0].strip().strip('"')
        named = [(a.split("=")[0].strip(), a.split("=", 1)[1] if "=" in a else "") for a in args[1:]]
        calls.append((name, [a for a, _ in named if a != "NAOK"], [v for a, v in named if a != "NAOK"]))
    return calls


def test_every_dot_c_call_matches_its_prototype():
    protos = prototypes()
    kinds = prototype_kinds()
    seen = set()
    n_args = n_known = 0
    for fn in sorted(os.listdir(os.path.join(ROOT, "R"))):
        if not fn.endswith(".R"):
            continue
        text = "\n".join(l.split("#")[0] for l in open(os.path.join(ROOT, "R", fn)).read().splitlines())
        for name, args, values in dot_c_calls(text):
            assert name in protos, (fn, name)
            want = kinds[name]
            assert "other" not in want, (fn, name, "has a parameter .C() cannot pass (char * / void **): bind it through a char ** / double variant")
            known = 0
            for arg, val, w in zip(args, values, want):
                k = r_kind(val)
                if k is not None:
                    known += 1
                    assert k == w, (fn, name, arg, val.strip(), "is passed as", k, "but the prototype takes", w)
            n_args += len(args)
            n_known += known
            assert len(args) == len(protos[name]), (fn, name, args, protos[name])
            assert args == protos[name], (fn, name, args, protos[name])      # same names in the same order as the prototype
            assert args[-1] == "status" or name == "nngp_last_error_r", (fn, name)
            seen.add(name)
    # the glue covers the entry points the reference's R code needs (INTEGRATION.md section 3)
    for need in ("nngp_ctx_create", "nngp_ctx_destroy", "nngp_factor_build", "nngp_loglik", "nngp_gibbs_sweep", "nngp_chain_run",
                 "nngp_regressors_set", "nngp_chain_run_regressors", "nngp_predict_sample", "nngp_field_init",
                 "nngp_host_find_ordered_nn", "nngp_host_greedy_coloring", "nngp_host_order_maxmin", "nngp_last_error_r", "nngp_chains_run",
                 "nngp_chains_run_regressors", "nngp_host_greedy_coloring_adj"):
        assert need in seen, need
    assert "nngp_last_error" not in seen          # char *: would be handed R's char ** (round-1 advisor finding)
    assert n_known >= 0.85 * n_args, (n_known, n_args)   # the kind check must actually cover the glue


def test_initialize_patch_applies_to_the_reference_and_calls_only_bound_wrappers():
    patch = os.path.join(ROOT, "R", "patches", "mcmc_nngp_initialize.patch")
    text = open(patch).read()
    glue = open(os.path.join(ROOT, "R", "nngp_b200.R")).read()
    added = [l[1:] for l in text.splitlines() if l.startswith("+") and not l.startswith("+++")]
    used = set(re.findall(r"\b(nngp_\w+)\(", "\n".join(added)))
    assert used >= {"nngp_find_ordered_nn", "nngp_greedy_coloring", "nngp_chain_context", "nngp_factor_build", "nngp_field_init", "nngp_field_get"}
    for f in used:
        assert re.search(rf"^{f}\s*=\s*function", glue, flags=re.M), f      # every wrapper the patch calls exists in R/nngp_b200.R
    ref = os.path.join(ROOT, "tests", "golden", "mcmc_nngp_initialize_excerpt.R")   # the reference's lines the patch touches
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "Scripts"))
        shutil.copy(ref, os.path.join(d, "Scripts", "mcmc_nngp_initialize.R"))
        r = subprocess.run(["patch", "-p0", "--dry-run", "-i", patch], cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        r = subprocess.run(["patch", "-p0", "-i", patch], cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        out = open(os.path.join(d, "Scripts", "mcmc_nngp_initialize.R")).read()
        assert "GpGp::vecchia_Linv" not in out and "naive_greedy_coloring" not in out and "nngp_field_init" in out


def test_dot_call_glue_compiles_against_the_r_api_it_uses():
    """R/r_glue.c (external-pointer contexts with a finalizer, long-vector outputs) against tests/r_stub/Rinternals.h: syntax, types
    and the argument counts of the library calls it makes; the registration table must list every SEXP entry point with its arity"""
    src = open(os.path.join(ROOT, "R", "r_glue.c")).read()
    r = subprocess.run(["gcc", "-fsyntax-only", "-Wall", "-Werror=implicit-function-declaration", "-Werror=incompatible-pointer-types", "-Werror=int-conversion",
                        "-I" + os.path.join(ROOT, "tests", "r_stub"), "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "R", "r_glue.c")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    defs = {name: len([a for a in args.split(",") if a.strip()]) for name, args in re.findall(r"^SEXP\s+(nngp_r_\w+)\s*\(([^)]*)\)\s*\{", src, flags=re.M)}
    table = {name: int(k) for name, k in re.findall(r'\{"(nngp_r_\w+)",\s*\(DL_FUNC\)&\w+,\s*(\d+)\}', src)}
    assert defs == table and len(defs) >= 4
    assert "R_RegisterCFinalizerEx" in src and "nngp_ctx_destroy" in src
