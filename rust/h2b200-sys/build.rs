//! Compiles halo2_scaffold_b200/csrc/*.cu with nvcc for sm_100a into a static library and links the CUDA runtime.
//! Equivalent to halo2_scaffold_b200/csrc/Makefile (which the Python/C++ tests use to build the shared library).
use std::env;
use std::path::PathBuf;
use std::process::Command;

fn main() {
    let manifest = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap());
    let csrc = manifest.join("../../halo2_scaffold_b200/csrc");
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let cuda = env::var("CUDA_HOME").unwrap_or_else(|_| "/usr/local/cuda".into());

    if env::var("CARGO_FEATURE_PREBUILT").is_ok() {
        let dir = env::var("H2B200_LIB_DIR").expect("feature `prebuilt` needs H2B200_LIB_DIR");
        println!("cargo:rustc-link-search=native={dir}");
        println!("cargo:rustc-link-lib=dylib=h2b200");
        return;
    }

    let sources = ["api.cu", "api_sets.cu", "api_srs.cu", "api_keygen.cu", "api_open.cu", "ntt.cu", "msm.cu", "testgen.cu", "g1gen.cu", "stage.cu", "scan.cu", "evaluate.cu", "srs.cu", "lookup.cu", "keygen.cu", "multiopen.cu"];
    let mut objects = Vec::new();
    for src in sources {
        let obj = out.join(src.replace(".cu", ".o"));
        let status = Command::new(format!("{cuda}/bin/nvcc"))
            .args(["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-c"])
            .arg(csrc.join(src))
            .arg("-o")
            .arg(&obj)
            .status()
            .expect("nvcc not found (set CUDA_HOME)");
        assert!(status.success(), "nvcc failed on {src}");
        objects.push(obj);
        println!("cargo:rerun-if-changed={}", csrc.join(src).display());
    }
    for hdr in ["common.h", "field.cuh", "ec.cuh", "field_asm.inc"] {
        println!("cargo:rerun-if-changed={}", csrc.join(hdr).display());
    }
    let lib = out.join("libh2b200.a");
    let status = Command::new("ar").arg("crs").arg(&lib).args(&objects).status().expect("ar");
    assert!(status.success());
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=static=h2b200");
    println!("cargo:rustc-link-search=native={cuda}/lib64");
    println!("cargo:rustc-link-lib=dylib=cudart");
    println!("cargo:rustc-link-lib=dylib=stdc++");
}
