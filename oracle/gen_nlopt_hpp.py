"""gen_nlopt_hpp.py <reference src/api dir> <output nlopt.hpp> -- the reference's C++ header generated the way its
cmake/generate-cpp.cmake:39-52 does: nlopt-in.hpp with the algorithm and result enums of nlopt.h spliced in at
GEN_ENUMS_HERE.  Used by `make refprog` (oracle/Makefile)."""
import re
import sys


def generate(api_dir, path):
    src = open(f"{api_dir}/nlopt-in.hpp").read().splitlines()
    hdr = open(f"{api_dir}/nlopt.h").read().splitlines()
    out = []
    for line in src:
        out.append(line)
        if "GEN_ENUMS_HERE" in line:
            out.append("  enum algorithm {")
            for h in hdr:
                if re.search(r"    NLOPT_[A-Z0-9_]+", h):
                    out.append(h.replace("NLOPT_", ""))
                    if "NLOPT_NUM_ALGORITHMS" in h:
                        out += ["  };", "  enum result {"]
                    elif "NLOPT_NUM_RESULTS" in h:
                        out.append("  };")
    with open(path, "w") as f:
        f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    generate(sys.argv[1], sys.argv[2])
