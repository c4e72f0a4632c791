// build.rs -- UNVERIFIED (no Rust toolchain in the build image).
// Compiles the sm_100a engine into a static library with nvcc and links it.
use std::{env, path::PathBuf, process::Command};

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let root = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap());
    let csrc = root.join("rust-msbwt_b200").join("csrc");
    let nvcc = env::var("NVCC").unwrap_or_else(|_| "nvcc".into());
    let mut objs = vec![];
    // the same list as rust-msbwt_b200/build.py SOURCES
    for f in ["capi.cu", "hostpath.cu", "kernels.cu", "quad_kernels.cu", "stats_kernels.cu", "wide_kernels.cu", "final_kernels.cu", "ext_kernels.cu",
              "loader.cu", "builder.cu", "pair_builder.cu", "quad_builder.cu", "oct_builder.cu", "fin_builder.cu", "bwt_build.cu", "bwt_merge.cu", "spectrum.cu", "unitigs.cu", "correct.cu"] {
        let obj = out.join(f).with_extension("o");
        let ok = Command::new(&nvcc)
            .args(["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
                   "-Xcompiler", "-fPIC", "-c", "-o"])
            .arg(&obj)
            .arg(csrc.join(f))
            .status()
            .expect("nvcc not found: this crate feature has no CPU fallback")
            .success();
        assert!(ok, "nvcc failed on {f}");
        println!("cargo:rerun-if-changed={}", csrc.join(f).display());
        objs.push(obj);
    }
    // the host-side 2-bit packer of the end-to-end path (plain C++, AVX2 behind a runtime check)
    let hp = out.join("hostpack.o");
    assert!(Command::new("g++").args(["-O3", "-std=c++17", "-fPIC", "-pthread", "-c", "-o"]).arg(&hp)
        .arg(csrc.join("hostpack.cpp")).status().expect("g++ not found").success());
    objs.push(hp);
    // the host codec (convert_to_vec / save_bwt_numpy: plain C++)
    let cd = out.join("codec.o");
    assert!(Command::new("g++").args(["-O3", "-std=c++17", "-fPIC", "-c", "-o"]).arg(&cd)
        .arg(csrc.join("codec.cpp")).status().expect("g++ not found").success());
    objs.push(cd);
    let lib = out.join("libmsbwt_b200.a");
    assert!(Command::new("ar").arg("crs").arg(&lib).args(&objs).status().unwrap().success());
    let cuda = env::var("CUDA_HOME").unwrap_or_else(|_| "/usr/local/cuda".into());
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-search=native={cuda}/lib64");
    println!("cargo:rustc-link-lib=static=msbwt_b200");
    println!("cargo:rustc-link-lib=dylib=cudart");
    println!("cargo:rustc-link-lib=dylib=stdc++");
}
