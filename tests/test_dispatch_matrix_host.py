"""Every kernel arm of libb2f's dispatch has a GPU case (no GPU needed).

The arms are read from the sources: the `case N:` lists and mode switches of b2f_ka.cu, b2f_kb.cu, b2f_kc.cu, b2f_kf.cu and
b2f_kg.cu, the per-size objects of the Makefile, the generic kernels launched in b2f_api.cu and the passes of b2f_kl.cu.
Each must be a key of test_gpu_dispatch_matrix.MATRIX, or be listed in NOT_BUILT with the reason it is never compiled.  A
new arm without a test fails here."""
import os
import re

from test_gpu_dispatch_matrix import CASES, MATRIX, derive_matrix

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "frb-baseband_b200", "csrc")
MODES = {"B2F_POL_P0": "P0", "B2F_POL_P1": "P1", "B2F_POL_I": "I", "B2F_POL_I2": "I2", "B2F_POL_PPQQ": "PPQQ",
         "B2F_POL_COHERENCE": "coherence", "B2F_POL_IQUV": "IQUV", "kModeSpectrum": "spectrum"}
_OFF = ("P0", "P1", "I2", "PPQQ")
_WHY = "round-2 kernels are built for I, coherence and IQUV only (Makefile B2F_KF_MAIN_MODES); the other products take path 0"
NOT_BUILT = {
    **{("kr", R, m): _WHY for R in (16, 32, 64, 128, 512) for m in _OFF},
    **{("kf", R, m): _WHY for R in (16, 32, 64, 128, 256, 512) for m in _OFF},
}


def src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def built_lines(text):
    """(line, built) for every line: built is False inside a preprocessor branch that the default build (the Makefile
    defines B2F_KF_MAIN_MODES, KFALL unset) compiles out.  Other conditions (B2F_PART, B2F_KF_PART) select between
    translation units that are all built, so their branches all count."""
    def off(cond):
        return bool(re.search(r"#\s*ifndef\s+B2F_KF_MAIN_MODES|!\s*defined\(B2F_KF_MAIN_MODES\)", cond))
    stack, out = [], []
    for line in text.splitlines():
        s = line.strip()
        if re.match(r"#\s*if", s):
            stack.append(off(s))
        elif re.match(r"#\s*elif", s):
            stack[-1] = off(s)
        elif re.match(r"#\s*else", s):
            stack[-1] = False
        elif re.match(r"#\s*endif", s):
            stack.pop()
        else:
            out.append((line, not any(stack)))
    return out


def function_body(text, signature):
    """Text of the function whose definition starts with `signature` (to its closing brace at column 0)."""
    i = text.index(signature)
    return text[i:text.index("\n}", i)]


def make_sizes(prefix):
    """The per-size objects the Makefile links: build/<prefix><N>.o -> [N]."""
    objs = re.search(r"^OBJS\s*:=(.*)$", src("Makefile"), re.M).group(1).split()
    return sorted(int(m.group(1)) for o in objs if (m := re.fullmatch(rf"build/{prefix}(\d+)\.o", o)))


def modes_in(text, call):
    """{(mode, built)} of the `case B2F_POL_x: return <call>` lines of a switch."""
    return {(MODES[m.group(1)], b) for line, b in built_lines(text) if (m := re.search(rf"case (\w+): return {call}", line))}


def parsed_arms():
    """{key: built} of every arm in the sources."""
    arms = {}

    def add(key, built=True):
        arms[key] = arms.get(key, False) or built

    ka = src("b2f_ka.cu")
    for nbit in make_sizes("ka"):
        for m in re.finditer(r"case (\d+): return go<\1, (true|false)>", ka):
            add(("ka", nbit, int(m.group(1)), "fwd" if m.group(2) == "true" else "full"))

    kb = src("b2f_kb.cu")
    kb_modes = modes_in(function_body(kb, "static cudaError_t by_mode("), "go<")
    kr_modes = modes_in(function_body(kb, "static cudaError_t by_mode_r("), "go_r<")
    for R in map(int, re.findall(r"case (\d+): return by_mode<", kb)):
        for mode, b in kb_modes:
            add(("kb", R, mode), b)
    for R in map(int, re.findall(r"case (\d+): return by_mode_r<", kb)):
        for mode, b in kr_modes:
            add(("kr", R, mode), b)

    for R in map(int, re.findall(r"case (\d+): return go<\1>", src("b2f_kc.cu"))):
        add(("kc_back", R))
        add(("kc_trials", R))

    kf = src("b2f_kf.cu")
    kfj_modes = modes_in(function_body(kf, "cudaError_t B2F_CAT(b2f_launch_kfj_, B2F_FR)(int mode, const FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm) {"), "go2<")
    kf_modes = modes_in(function_body(kf, "cudaError_t B2F_CAT(b2f_launch_kf_, B2F_FR)("), "go<")
    for R in make_sizes("kfj"):
        for mode, b in kfj_modes:
            add(("kfj", R, mode), b)
    for R in make_sizes("kf"):
        for mode, b in kf_modes:
            add(("kf", R, mode), b)

    kg = src("b2f_kg.cu")
    row_modes = modes_in(kg, "row_go<")
    col_nbits = sorted({int(n) for n in re.findall(r"col_go<(\d+)>\(", kg)})
    for lg in make_sizes("kg"):
        for mode, b in row_modes:
            add(("kgt_row", lg, mode), b)
        for nbit in col_nbits:
            add(("kgt_col", lg, nbit))

    api = src("b2f_api.cu")
    for nbit in re.findall(r"kg_column_pass<(\d+)><<<", api):
        add(("kg_col", int(nbit)))
    for cpt, arg in re.findall(r"kg_row_pass<(\d+)><<<[^;]*>>>\((\w+)\);", api):
        add(("kg_row", int(cpt), {"kv": "volt", "kg": "detect"}[arg]))
    if re.search(r"kx_dedisp_generic<<<", api):
        add(("kx",))

    kl = src("b2f_kl.cu")
    for load in re.findall(r"run_pass<kLoad(\w+)>\(", kl):
        add(("kl_pass", load.lower()))
    detect = function_body(kl, "__global__ void __launch_bounds__(256) kl_detect(")
    for m in re.findall(r"case (B2F_POL_\w+):", detect):
        add(("kl_detect", MODES[m]))
    if "default:" in detect:                      # the default arm accumulates I, 2 Re, 2 Im, PP - QQ: IQUV
        add(("kl_detect", "IQUV"))
    return arms


def test_parser_sees_every_family():
    """The parser finds the arms it is meant to find (a changed source layout must not make this test vacuous)."""
    arms = parsed_arms()
    fams = {k[0] for k in arms}
    assert fams == {"ka", "kb", "kr", "kc_back", "kc_trials", "kf", "kfj", "kgt_row", "kgt_col", "kg_col", "kg_row", "kx", "kl_pass",
                    "kl_detect"}, fams
    assert ("kc_back", 16) in arms and ("kg_row", 8, "volt") in arms and ("kgt_row", 13, "IQUV") in arms and ("kfj", 32, "I") in arms
    assert len([k for k in arms if k[0] == "kb"]) == 6 * 8 and len([k for k in arms if k[0] == "ka"]) == 3 * 6 * 2


def test_every_built_arm_has_a_case():
    arms = parsed_arms()
    built = {k for k, b in arms.items() if b}
    missing = sorted(map(str, built - set(MATRIX)))
    assert not missing, f"{len(missing)} kernel arms have no case in test_gpu_dispatch_matrix: {missing}"


def test_arms_compiled_out_are_listed():
    arms = parsed_arms()
    off = {k for k, b in arms.items() if not b}
    assert off == set(NOT_BUILT), (sorted(map(str, off - set(NOT_BUILT))), sorted(map(str, set(NOT_BUILT) - off)))
    assert not off & set(MATRIX)


def test_matrix_keys_have_cases():
    arms = parsed_arms()
    for key, ids in MATRIX.items():
        assert ids, key
        assert all(i in CASES for i in ids), (key, [i for i in ids if i not in CASES])
        assert key in arms or key[0] == "kt", f"{key}: not an arm of the sources"


def test_matrix_is_what_the_cases_reach():
    """MATRIX is the selection rule applied to CASES: a case added, removed or changed shows in the map."""
    derived = derive_matrix()
    assert set(MATRIX) == set(derived), (sorted(map(str, set(MATRIX) - set(derived))), sorted(map(str, set(derived) - set(MATRIX))))
    for key in MATRIX:
        assert MATRIX[key] == derived[key], key
