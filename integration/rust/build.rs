// build.rs -- po-rrt crate root.  Without `--features b200` it does nothing.  With it, the CUDA sources of po_rrt_b200/csrc are
// compiled for sm_100a (B200) into libporrt_b200.so next to the other build artefacts and linked as a dylib.
// (Written against the reference tree; cargo / rustc are not part of the image this repository is built in, so this file has
// not been run there -- tests/c_abi_harness.c and po_rrt_b200/api.py exercise the same library from C and Python.)
use std::path::PathBuf;
use std::process::Command;

const CU_SOURCES: &[&str] = &[
    "ctx.cu", "map.cu", "edge3.cu", "nn.cu", "nn_tile.cu", "graph.cu", "colsolve.cu", "sssp_frontier.cu", "belief_tables.cu", "belief_explicit.cu",
    "mmprm.cu", "refine.cu", "comm.cu", "host_side.cu", "formats.cu", "diag.cu", "pto_grow.cu",
];
const HEADERS: &[&str] = &[
    "common.cuh", "colsolve.cuh", "belief_tables.cuh", "sssp_frontier.cuh", "map_dev.cuh", "edge_common.cuh", "nn_dev.cuh", "pcg64.h",
];

fn main() {
    println!("cargo:rerun-if-env-changed=PORRT_B200_SRC");
    if std::env::var("CARGO_FEATURE_B200").is_err() {
        return;
    }
    // where the po_rrt_b200 checkout lives (a git submodule under vendor/ by default)
    let src_root = PathBuf::from(std::env::var("PORRT_B200_SRC").unwrap_or_else(|_| "vendor/po_rrt_b200".to_string()));
    let csrc = src_root.join("po_rrt_b200").join("csrc");
    let out = PathBuf::from(std::env::var("OUT_DIR").unwrap());
    let nvcc = std::env::var("NVCC").unwrap_or_else(|_| "nvcc".to_string());
    let mut objects = Vec::new();
    for s in CU_SOURCES {
        let src = csrc.join(s);
        println!("cargo:rerun-if-changed={}", src.display());
        let obj = out.join(s.replace(".cu", ".o"));
        // -fmad=false: Rust never contracts a * b + c; the bit-exactness contract depends on it (DESIGN.md section 4)
        let status = Command::new(&nvcc)
            .args(["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false"])
            .args(["-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off", "-c"])
            .arg(&src)
            .arg("-o")
            .arg(&obj)
            .status()
            .expect("nvcc not found (set NVCC)");
        assert!(status.success(), "nvcc failed on {}", src.display());
        objects.push(obj);
    }
    for h in HEADERS {
        println!("cargo:rerun-if-changed={}", csrc.join(h).display());
    }
    println!("cargo:rerun-if-changed={}", src_root.join("include").join("porrt_b200.h").display());
    let so = out.join("libporrt_b200.so");
    let status = Command::new(&nvcc)
        .args(["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o"])
        .arg(&so)
        .args(&objects)
        .args(["-lcudart_static", "-lpthread", "-ldl", "-lrt"])
        .status()
        .expect("nvcc not found (set NVCC)");
    assert!(status.success(), "linking libporrt_b200.so failed");
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=dylib=porrt_b200");
    println!("cargo:rustc-link-arg=-Wl,-rpath,{}", out.display());
}
