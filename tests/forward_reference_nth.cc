// tests/forward_reference_nth.cc -- TEST INFRASTRUCTURE ONLY: the C++ standard library's own std::nth_element on floats, as
// CachedForwardInterpolation's median calls it, for tests/forward_reference.py.  Compiled on first use with the system g++.
#include <algorithm>
#include <cstddef>

extern "C" void ref_nth_element(float* v, std::size_t nth, std::size_t n)
{
    std::nth_element(v, v + nth, v + n);
}
