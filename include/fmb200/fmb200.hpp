// fmb200/fmb200.hpp -- umbrella header of the C++ host side (the counterpart of fmindex-collection/fmindex-collection.h).
#pragma once
#include "adapt.hpp"
#include "host_mirror.hpp"
#include "index.hpp"
#include "multi.hpp"
#include "search.hpp"
#include "search_scheme.hpp"
#include "smem.hpp"
#include "io.hpp"
