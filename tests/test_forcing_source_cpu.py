"""CPU: forcing sources compile for sm_100a through nsb_check_forcing_source (NVRTC, no GPU), and the ones that break the
source contract of include/nsb200.h are rejected with NVRTC's log."""
import re

import pytest

from tests.forcing_sources import IDENTITY, MANUFACTURED, SCALED, SMOOTH, ZERO

GOOD = dict(smooth=SMOOTH, manufactured=MANUFACTURED, identity=IDENTITY, zero=ZERO, scaled=SCALED)

SIG = "__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f)"
BAD = {
    "missing": ("__device__ void my_forcing(const double* x, double t, const double* prm, double* f) { f[0] = x[0]; }\n",
                r"nsb_forcing"),
    "float_time": ("__device__ void nsb_forcing(const double* x, float t, const double* prm, double* f) { f[0] = t; }\n",
                   r"nsb_forcing must be declared as"),
    "returns_double": ("__device__ double nsb_forcing(const double* x, double t, const double* prm, double* f) { return x[0]; }\n",
                       r"nsb_forcing must be declared as"),
    "two_arguments": ("__device__ void nsb_forcing(const double* x, double* f) { f[0] = x[0]; }\n", r"nsb_forcing"),
    "host_only": ("void nsb_forcing(const double* x, double t, const double* prm, double* f) { f[0] = x[0]; }\n",
                  r"__host__"),
    "include": ("#include <cmath>\n" + SIG + " { f[0] = x[0]; }\n", r"nsb_forcing\.cu\(1\).*cmath"),
}


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("name", list(GOOD))
def test_forcing_sources_compile(nsb, dim, name):
    nsb.check_forcing_source(dim, GOOD[name])


@pytest.mark.parametrize("dim", [2, 3])
def test_syntax_error_names_the_line(nsb, dim):
    src = SIG + " {\n  f[0] = x[0];\n  f[1] = x[1]\n  f[0] += 1.0;\n}\n"       # missing ';' at the end of line 3
    with pytest.raises(nsb.NsbError) as e:
        nsb.check_forcing_source(dim, src)
    msg = str(e.value)
    assert re.search(r"nsb_forcing\.cu\((3|4)\): error", msg), msg
    assert "f[0] += 1.0" in msg or "f[1] = x[1]" in msg, msg


@pytest.mark.parametrize("name", list(BAD))
def test_contract_violations_are_rejected(nsb, name):
    src, pattern = BAD[name]
    with pytest.raises(nsb.NsbError) as e:
        nsb.check_forcing_source(3, src)
    assert re.search(pattern, str(e.value), re.S), str(e.value)


def test_check_forcing_source_return_codes(nsb):
    import ctypes as C
    L = nsb.lib()
    assert L.nsb_check_forcing_source(3, SMOOTH.encode(), None, C.c_size_t(0)) == 0
    buf = C.create_string_buffer(16)                          # the log is truncated to the buffer and NUL-terminated
    assert L.nsb_check_forcing_source(3, b"nonsense", buf, C.c_size_t(len(buf))) < 0
    assert len(buf.value) == 15
    buf = C.create_string_buffer(256)
    assert L.nsb_check_forcing_source(4, SMOOTH.encode(), buf, C.c_size_t(len(buf))) < 0
    assert b"dim" in buf.value
    assert L.nsb_check_forcing_source(2, None, buf, C.c_size_t(len(buf))) < 0


def test_device_forcing_has_no_host_evaluation(tmp_path):
    """DeviceForcing<dim>::value throws: the term is evaluated on the GPU only, never silently on the host."""
    import os
    import subprocess
    from tests.conftest import ROOT
    src = tmp_path / "df.cpp"
    src.write_text(r'''
#include <iostream>
#include "navier_stokes.hpp"
int main() {
  nsb_host::DeviceForcing<3> f("__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {}", {1.0});
  nsb_host::Vector<double> v(4);
  try { f.vector_value(nsb_host::Point<3>(0.1, 0.2, 0.3), v); } catch (const std::logic_error& e) { std::cout << e.what() << std::endl; }
  try { nsb_host::DeviceForcing<2> g("", std::vector<double>(17, 0.0)); } catch (const std::invalid_argument& e) { std::cout << e.what() << std::endl; }
  return f.params().size() == 1 ? 0 : 1;
}
''')
    exe = tmp_path / "df"
    host = os.path.join(ROOT, "navier-stokes_equations_b200", "host")
    r = subprocess.run(["g++", "-std=c++17", "-I", host, "-o", str(exe), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "evaluated on the GPU only" in r.stdout and "at most 16 parameters" in r.stdout, r.stdout
