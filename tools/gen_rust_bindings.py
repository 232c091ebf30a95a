"""Regenerates include/onb_sys.rs (the unbuilt Rust bindings of the C ABI) from include/onb.h:

    python tools/gen_rust_bindings.py
"""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TMAP = {'int32_t': 'i32', 'uint32_t': 'u32', 'int64_t': 'i64', 'uint64_t': 'u64', 'double': 'f64', 'float': 'f32', 'uint8_t': 'u8',
        'uint16_t': 'u16', 'onb_action': 'u16', 'void': 'c_void', 'char': 'c_char', 'onb_ctx': 'onb_ctx', 'onb_config': 'onb_config',
        'onb_state': 'onb_state', 'onb_tree_dump': 'onb_tree_dump', 'onb_selfplay_config': 'onb_selfplay_config',
        'onb_selfplay_result': 'onb_selfplay_result', 'onb_agent': 'onb_agent', 'onb_fight_result': 'onb_fight_result',
        'onb_actor': 'onb_actor', 'onb_actor_view': 'onb_actor_view', 'onb_fight_statistics': 'onb_fight_statistics', 'onb_comm': 'onb_comm', 'onb_replay': 'onb_replay',
        'onb_gumbel_config': 'onb_gumbel_config', 'int16_t': 'i16', 'onb_tb_class': 'onb_tb_class'}
I32_PREFIXES = ('ONB_E_', 'ONB_BUF', 'ONB_STAT', 'ONB_RESULT', 'ONB_POLICY', 'ONB_EVAL', 'ONB_AGENT', 'ONB_NET_', 'ONB_SELFTEST', 'ONB_ALPHABETA', 'ONB_TB_MAX')
I32_NAMES = ('ONB_VERSION', 'ONB_OK', 'ONB_RED', 'ONB_BLUE', 'ONB_PAWN', 'ONB_KING')
STRUCTS = '''#[repr(C)]
pub struct onb_ctx { _private: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy, Default, Debug, PartialEq, Eq)]
pub struct onb_state {
    pub pawns: [u32; 2],
    pub kings: [u32; 2],
    pub cards: [u8; 5],
    pub side: u8,
    pub result: u8,
    pub flags: u8,
}

#[repr(C)]
pub struct onb_config {
    pub device: i32,
    pub flags: u32,
    pub n_games: i64,
    pub game_id_base: u64,
    pub seed: u64,
    pub stream: *mut c_void,
    pub mcts_max_sims: u32,
    pub mcts_node_cap: u32,
    pub alloc_planes: u32,
    pub reserved: u32,
}

#[repr(C)]
pub struct onb_tree_dump {
    pub visits: *mut u32,
    pub reward: *mut f64,
    pub prior: *mut f64,
    pub action: *mut u16,
    pub parent: *mut i32,
    pub first_child: *mut u32,
    pub n_child: *mut u32,
    pub flags: *mut u8,
}

#[repr(C)]
pub struct onb_selfplay_config {
    pub c_puct: f64,
    pub sims: u32,
    pub evaluator: i32,
    pub n_games: i64,
    pub max_plies: u32,
    pub train: i32,
    pub noise_seed: u64,
    pub sample_cap: i64,
}

#[repr(C)]
pub struct onb_selfplay_result {
    pub n_samples: i64,
    pub n_valid: i64,
    pub n_games: i64,
    pub plies_run: i64,
    pub truncated: i32,
    pub reserved: i32,
    pub planes: *mut f32,
    pub pi: *mut f32,
    pub z: *mut f32,
    pub color: *mut u8,
    pub serial: *mut i64,
    pub valid_idx: *mut i64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct onb_gumbel_config {
    pub enabled: i32,
    pub max_considered: u32,
    pub c_visit: f64,
    pub c_scale: f64,
    pub gumbel_scale: f64,
    pub seed: u64,
    pub step0: u32,
    pub reserved: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct onb_tb_class {
    pub entries: i64,
    pub wins: i64,
    pub losses: i64,
    pub draws: i64,
    pub invalid: i64,
    pub max_win: i32,
    pub max_loss: i32,
    pub iterations: i32,
    pub solved: i32,
    pub examined: i64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct onb_agent {
    pub kind: i32,
    pub evaluator: i32,
    pub net_slot: i32,
    pub sims: u32,
    pub c: f64,
    pub min_node_visits: u32,
    pub reserved: u32,
}

#[repr(C)]
pub struct onb_actor { _private: [u8; 0] }

#[repr(C)]
pub struct onb_comm { _private: [u8; 0] }

#[repr(C)]
pub struct onb_replay { _private: [u8; 0] }

#[repr(C)]
pub struct onb_actor_view {
    pub first: i64,
    pub count: i64,
    pub actions: *mut u16,
    pub masks: *mut u32,
    pub done: *mut u32,
    pub stats: *mut u64,
}

#[repr(C)]
pub struct onb_fight_result {
    pub a_wins: i64,
    pub b_wins: i64,
    pub draws: i64,
    pub plies_run: i64,
    pub results: *mut u8,
    pub moves_chosen: i64,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct onb_fight_statistics {
    pub n_games: i64,
    pub wins: i64,
    pub loses: i64,
    pub draws: i64,
    pub color_wins: [i64; 2],
    pub color_loses: [i64; 2],
    pub color_draws: [i64; 2],
    pub winrate: f64,
    pub color_winrate: [f64; 2],
    pub rating_a: f64,
    pub rating_b: f64,
}
'''


def conv_type(t):
    t = t.strip()
    const = 'const ' in t
    t = t.replace('const', '').strip()
    ptr = t.count('*')
    r = TMAP[t.replace('*', '').strip()]
    for _ in range(ptr):
        r = ('*const ' if const else '*mut ') + r
    return r


def main():
    hdr = open(os.path.join(ROOT, 'include', 'onb.h')).read()
    body = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    decls = re.findall(r"ONB_API\s+([^;]+?)\s+(onb_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", body, flags=re.S)
    fns = []
    for ret, name, args in decls:
        args = ' '.join(args.split())
        params = []
        if args and args != 'void':
            for a in args.split(','):
                m = re.match(r"(.+?)([A-Za-z_][A-Za-z0-9_]*)(\[[^\]]*\])?$", a.strip())
                typ = m.group(1) + ('*' if m.group(3) else '')
                params.append("%s: %s" % (m.group(2), conv_type(typ)))
        fns.append("    pub fn %s(%s) -> %s;" % (name, ', '.join(params), conv_type(ret)))
    lines = ['// onb_sys.rs -- raw Rust bindings of include/onb.h (libonb.so), GENERATED by tools/gen_rust_bindings.py.',
             '// NOT BUILT in this repository: the image has no cargo/rustc. A maintainer of cyoq/onitama-alphazero would drop this file into',
             '// alphazero-training/src/ and link with `cargo:rustc-link-lib=dylib=onb` (INTEGRATION.md section 1).',
             '// tests/test_abi_cpu.py checks that every symbol declared in onb.h is bound here.',
             '#![allow(non_camel_case_types, dead_code)]', 'use std::os::raw::{c_char, c_void};', '']
    for k, v in re.findall(r"#define (ONB_[A-Z0-9_]+) (\(?-?\d+u?\)?)\s", body):
        v = v.strip('()').rstrip('u')
        if k in I32_NAMES or k.startswith(I32_PREFIXES):
            lines.append("pub const %s: i32 = %s;" % (k, v))
        elif k.startswith(('ONB_OUT', 'ONB_HOST')):
            lines.append("pub const %s: u32 = %s;" % (k, v))
    lines += ['pub const ONB_ACTION_NONE: u16 = 0xFFFF;', 'pub const ONB_TB_NONE: i16 = -32768;', '',
              '/// action code: to | from << 5 | used_card_idx << 10 | piece << 12 | pass << 13',
              'pub const fn onb_action(card_idx: u16, from: u16, to: u16, piece: u16) -> u16 { to | (from << 5) | (card_idx << 10) | (piece << 12) }',
              'pub const fn onb_action_pass(card_idx: u16) -> u16 { (card_idx << 10) | (1 << 13) }', '', STRUCTS,
              '#[link(name = "onb")]', 'extern "C" {'] + fns + ['}', '']
    open(os.path.join(ROOT, 'include', 'onb_sys.rs'), 'w').write('\n'.join(lines))
    print(len(fns), "functions bound")


if __name__ == '__main__':
    main()
